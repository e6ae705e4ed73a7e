"""Element-partitioned multi-GPU assembly: one process per GPU, interface rows summed over NCCL.

SURVEY.md section 8(e).  Elements are split across ranks; every rank assembles its own elements into
a local CSR with the same deterministic kernels as the single-GPU path.  A global row (DOF) that
is touched by elements of several ranks is OWNED by the lowest such rank; the other ranks send
their partial row sums (matrix entries and load entry) to the owner, which adds them in fixed
rank order.  Only those interface rows travel: for horizontal strips of the config-2 mesh that is
one vertex row (~14 k matrix entries + 2 k load entries, ~130 KB) per cut.

Set-up (integer, one-time, `torch.distributed` collectives on index tensors):
  1. owner / multiplicity of every global vertex by all-reduce(MIN / SUM);
  2. every rank tells each owner which (row, col) keys it will contribute; the owner adds columns
     it does not touch itself as ghost DOFs so its rows carry the full global pattern;
  3. both sides translate the agreed key list into positions in their own CSR value arrays.
Per assembly: pack (tfem_iface_pack) -> batched isend/irecv -> unpack-add (tfem_iface_unpack_add).
"""

from __future__ import annotations

import os
from dataclasses import dataclass
from typing import Callable, Dict, Optional

import torch
import torch.distributed as dist

from . import csr as csr_mod


@dataclass
class ExchangeOps:
    """How interface entries are gathered / accumulated (CUDA kernels in production)."""

    pack: Callable[[torch.Tensor, torch.Tensor], torch.Tensor]  # (src, idx) -> src[idx]
    unpack_add: Callable[[torch.Tensor, torch.Tensor, torch.Tensor], None]  # dst[idx] += buf
    pack_into: Callable[[torch.Tensor, torch.Tensor, torch.Tensor], None] = None  # out[:] = src[idx]

    def __post_init__(self):
        if self.pack_into is None:
            self.pack_into = lambda out, src, idx: out.copy_(self.pack(src, idx))


def cuda_exchange_ops() -> ExchangeOps:
    from . import ops

    # the per-step calls go straight to the C ABI (a few microseconds of host time each)
    return ExchangeOps(pack=ops.gather, unpack_add=ops.unpack_add_raw, pack_into=ops.pack_into_raw)


def _exchange_variable(send: Dict[int, torch.Tensor], rank: int, world: int, device, dtype, group) -> Dict[int, torch.Tensor]:
    """Every rank sends `send[peer]` (1-D, any length) to `peer`; returns what each peer sent us."""
    counts = torch.zeros(world, dtype=torch.int64, device=device)
    for peer, t in send.items():
        counts[peer] = t.numel()
    table = [torch.zeros(world, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(table, counts, group=group)
    incoming = {peer: int(table[peer][rank]) for peer in range(world) if peer != rank and int(table[peer][rank]) > 0}
    recv = {peer: torch.empty(n, dtype=dtype, device=device) for peer, n in incoming.items()}
    ops_list = []
    for peer in sorted(set(send) | set(recv)):
        # lower rank sends first: a fixed global order keeps blocking back-ends deadlock-free
        if peer in send and send[peer].numel() > 0:
            ops_list.append(dist.P2POp(dist.isend, send[peer].contiguous(), peer, group=group))
        if peer in recv:
            ops_list.append(dist.P2POp(dist.irecv, recv[peer], peer, group=group))
    if ops_list:
        for work in dist.batch_isend_irecv(ops_list):
            work.wait()
    return recv


class InterfacePlan:
    """Who owns which rows and where interface contributions sit in the local arrays."""

    def __init__(self, elem_global_conn: torch.Tensor, n_global: int, rank: int, world: int, group=None):
        device = elem_global_conn.device
        conn = elem_global_conn.reshape(-1, 3).long()
        self.rank, self.world, self.group, self.n_global = rank, world, group, n_global

        touched = torch.unique(conn)
        owner = torch.full((n_global,), world, dtype=torch.int32, device=device)
        owner[touched] = rank
        dist.all_reduce(owner, op=dist.ReduceOp.MIN, group=group)
        mult = torch.zeros(n_global, dtype=torch.int32, device=device)
        mult[touched] = 1
        dist.all_reduce(mult, op=dist.ReduceOp.SUM, group=group)
        self.owner_of_touched = owner[touched]
        self.interface_global = touched[mult[touched] > 1]

        # keys (row, col) of our COO whose row belongs to another rank, per owner
        rows = conn[:, [0, 1, 2, 0, 1, 2, 0, 1, 2]].reshape(-1)
        cols = conn.repeat_interleave(3, dim=1).reshape(-1)
        row_owner = owner[rows]
        foreign = row_owner != rank
        keys = torch.unique(rows[foreign] * n_global + cols[foreign])
        key_owner = owner[torch.div(keys, n_global, rounding_mode="floor")]
        self.send_keys = {int(o): keys[key_owner == o] for o in torch.unique(key_owner).tolist()}
        self.recv_keys = _exchange_variable(self.send_keys, rank, world, device, torch.int64, group)

        # ghost DOFs: columns of received keys that none of our own elements touches
        ghosts = [torch.empty(0, dtype=torch.int64, device=device)]
        for k in self.recv_keys.values():
            c = k % n_global
            ghosts.append(c[~torch.isin(c, touched)])
        self.local_to_global = torch.unique(torch.cat([touched, *ghosts]))
        self.n_local = int(self.local_to_global.numel())
        self.n_ghost = self.n_local - int(touched.numel())
        self.dof_conn = torch.searchsorted(self.local_to_global, conn).to(torch.int32)
        self.owned_rows = owner[self.local_to_global] == rank  # rows complete on this rank after exchange
        self.extra_keys = self._to_local_keys(torch.cat(list(self.recv_keys.values()))) if self.recv_keys else None

    def _to_local_keys(self, global_keys: torch.Tensor) -> torch.Tensor:
        r = torch.div(global_keys, self.n_global, rounding_mode="floor")
        c = global_keys - r * self.n_global
        return torch.searchsorted(self.local_to_global, r) * self.n_local + torch.searchsorted(self.local_to_global, c)

    def bind(self, pattern: csr_mod.CsrPattern):
        """Positions of every exchanged entry in this rank's CSR value / load arrays."""

        def positions(global_keys):
            local = self._to_local_keys(global_keys)
            pos = torch.searchsorted(pattern.keys, local)
            if not bool((pattern.keys[pos.clamp_max(pattern.nnz - 1)] == local).all()):
                raise RuntimeError("interface key missing from the local CSR pattern")
            rows_g = torch.unique(torch.div(global_keys, self.n_global, rounding_mode="floor"))
            return pos.to(torch.int32), torch.searchsorted(self.local_to_global, rows_g).to(torch.int32)

        self.send_idx = {peer: positions(k) for peer, k in self.send_keys.items()}
        self.recv_idx = {peer: positions(k) for peer, k in self.recv_keys.items()}
        return self


class InterfaceExchange:
    """Per-assembly exchange: pack -> isend/irecv -> unpack-add in ascending peer order."""

    def __init__(self, plan: InterfacePlan, exchange_ops: Optional[ExchangeOps] = None):
        self.plan = plan
        self.ops = exchange_ops or cuda_exchange_ops()
        self.bytes_sent = 0

    def __call__(self, values: Optional[torch.Tensor], load: Optional[torch.Tensor]):
        plan = self.plan
        load_flat = load.reshape(-1) if load is not None else None
        send_bufs, recv_bufs, p2p = {}, {}, []
        for peer in sorted(set(plan.send_idx) | set(plan.recv_idx)):
            if peer in plan.send_idx:
                vi, ri = plan.send_idx[peer]
                parts = []
                if values is not None:
                    parts.append(self.ops.pack(values, vi))
                if load_flat is not None:
                    parts.append(self.ops.pack(load_flat, ri))
                send_bufs[peer] = torch.cat(parts)
                self.bytes_sent += send_bufs[peer].numel() * send_bufs[peer].element_size()
                p2p.append(dist.P2POp(dist.isend, send_bufs[peer], peer, group=plan.group))
            if peer in plan.recv_idx:
                vi, ri = plan.recv_idx[peer]
                n = (vi.numel() if values is not None else 0) + (ri.numel() if load_flat is not None else 0)
                ref = values if values is not None else load_flat
                recv_bufs[peer] = torch.empty(n, dtype=ref.dtype, device=ref.device)
                p2p.append(dist.P2POp(dist.irecv, recv_bufs[peer], peer, group=plan.group))
        if p2p:
            for work in dist.batch_isend_irecv(p2p):
                work.wait()
        for peer in sorted(recv_bufs):  # fixed order -> bitwise reproducible sums
            vi, ri = plan.recv_idx[peer]
            buf = recv_bufs[peer]
            offset = 0
            if values is not None:
                self.ops.unpack_add(values, vi, buf[: vi.numel()].contiguous())
                offset = vi.numel()
            if load_flat is not None:
                self.ops.unpack_add(load_flat, ri, buf[offset:].contiguous())


def strip_mesh(nx: int, ny: int, rank: int, world: int, jitter: float = 0.25, seed: int = 1234):
    """Rank `rank`'s horizontal strip of the `nx` x `ny*world` structured mesh on [0,1]x[0,world].

    Returns (mesh dict in local numbering, global vertex id of local vertex 0, n_global)."""
    from . import meshgen

    mesh = meshgen.structured_rectangle(nx, ny, 0.0, 1.0, float(rank), float(rank + 1), jitter=jitter, seed=seed + rank, topology=False)
    offset = rank * ny * (nx + 1)
    n_global = (nx + 1) * (ny * world + 1)
    return mesh, offset, n_global


class FusedExchange:
    """Interface exchange over ONE device buffer holding `[csr values | load vector]`.

    Every rank packs ALL its outgoing interface entries (for every owner, ascending) with one gather
    kernel into a fixed-size slot of a send buffer; one `all_gather` moves the slots (interfaces are a
    few hundred KB, so the redundancy is irrelevant and a single collective keeps the host cost of a
    step far below the assembly kernel's run time); each owner then adds the slices addressed to it,
    in ascending peer order, with one add kernel per peer.  Nothing synchronises with the host, so
    the whole exchange can sit on a side stream while the interior tiles are being assembled."""

    def __init__(self, plan: InterfacePlan, nnz: int, dtype: torch.dtype, device, exchange_ops: Optional[ExchangeOps] = None):
        self.plan = plan
        self.ops = exchange_ops or cuda_exchange_ops()
        world, rank = plan.world, plan.rank
        combine = lambda pair: torch.cat([pair[0], pair[1] + nnz]).to(torch.int32)  # noqa: E731
        owners = sorted(plan.send_idx)
        pieces = [combine(plan.send_idx[o]) for o in owners]
        self.send_idx = torch.cat(pieces).contiguous() if pieces else torch.zeros(0, dtype=torch.int32, device=device)
        # table[r, o] = (offset, length) of rank r's entries for owner o inside r's slot
        table = torch.zeros((world, 2), dtype=torch.int64, device=device)
        offset = 0
        for o, piece in zip(owners, pieces):
            table[o, 0], table[o, 1] = offset, piece.numel()
            offset += piece.numel()
        tables = [torch.zeros_like(table) for _ in range(world)]
        dist.all_gather(tables, table, group=plan.group)
        slot = torch.tensor([offset], dtype=torch.int64, device=device)
        dist.all_reduce(slot, op=dist.ReduceOp.MAX, group=plan.group)
        self.slot = max(int(slot.item()), 1)
        self.send_buf = torch.zeros(self.slot, dtype=dtype, device=device)
        self.gathered = torch.zeros((world, self.slot), dtype=dtype, device=device)
        self.recv = []  # (peer, local positions, offset, length), ascending peer
        for peer in sorted(plan.recv_idx):
            off, length = int(tables[peer][rank, 0]), int(tables[peer][rank, 1])
            idx = combine(plan.recv_idx[peer]).contiguous()
            assert idx.numel() == length, "interface key lists disagree between sender and owner"
            self.recv.append((peer, idx, off, length))
        self.peers = sorted(set(owners) | {p for p, *_ in self.recv})
        self.bytes_per_exchange = self.send_idx.numel() * self.send_buf.element_size()
        self.n_kernels = (1 if self.send_idx.numel() else 0) + len(self.recv)
        self.flat_gather = dist.get_backend(plan.group) == "nccl"

    def __call__(self, buffer: torch.Tensor):
        self.pack(buffer)
        self.gather_add(buffer)

    def pack(self, buffer: torch.Tensor):
        if self.send_idx.numel():
            self.ops.pack_into(self.send_buf[: self.send_idx.numel()], buffer, self.send_idx)

    def gather_add(self, buffer: torch.Tensor):
        if self.flat_gather:
            dist.all_gather_into_tensor(self.gathered, self.send_buf, group=self.plan.group)
        else:  # gloo (CPU tests) has no flat all-gather
            dist.all_gather(list(self.gathered.unbind(0)), self.send_buf, group=self.plan.group)
        for peer, idx, off, length in self.recv:  # ascending peer order -> bitwise reproducible sums
            self.ops.unpack_add(buffer, idx, self.gathered[peer, off : off + length])


class PeerExchange:
    """Interface exchange over NVLink peer memory (torch symmetric memory), no collective kernel.

    Every rank owns a receive buffer that its peers have mapped.  Per assembly the sender's pack
    kernel (`tfem_iface_pack`) gathers the interface entries of `[csr values | load]` and stores them
    STRAIGHT INTO THE OWNER'S BUFFER over NVLink, then raises a signal in the owner's signal pad;
    the owner waits for the signal on its side stream, adds the slice (`tfem_iface_unpack_add`,
    ascending peer order, so sums are bitwise reproducible) and hands the buffer back with a second
    signal.  Receive buffers alternate between two halves by step parity, so a sender never
    overwrites data its owner has not added yet.  All kernels are a single small CTA-group each
    and fit in the CTA slots the persistent interior launch leaves free (`reserve_ctas`), which a
    NCCL collective kernel does not: behind a persistent grid it would only start when the grid ends."""

    DATA, FREE = 0, 2  # signal channels: DATA + parity, FREE + parity

    def __init__(self, plan: InterfacePlan, nnz: int, dtype: torch.dtype, device, exchange_ops: Optional[ExchangeOps] = None,
                 timeout_ms: int = 20000):
        import torch.distributed._symmetric_memory as symm_mem

        self.plan = plan
        self.ops = exchange_ops or cuda_exchange_ops()
        self.timeout_ms = timeout_ms
        world, rank = plan.world, plan.rank
        group = plan.group if plan.group is not None else dist.group.WORLD
        combine = lambda pair: torch.cat([pair[0], pair[1] + nnz]).to(torch.int32).contiguous()  # noqa: E731
        sends = [(o, combine(plan.send_idx[o])) for o in sorted(plan.send_idx)]
        recvs = [(p, combine(plan.recv_idx[p])) for p in sorted(plan.recv_idx)]
        # where each sender's slice starts inside MY buffer; every rank learns its offsets at its owners
        offsets = torch.zeros(world, dtype=torch.int64, device=device)
        lengths = torch.zeros(world, dtype=torch.int64, device=device)
        used = 0
        for p, idx in recvs:
            offsets[p], lengths[p] = used, idx.numel()
            used += idx.numel()
        table = [torch.zeros(2 * world, dtype=torch.int64, device=device) for _ in range(world)]
        dist.all_gather(table, torch.cat([offsets, lengths]), group=group)
        cap = torch.tensor([used], dtype=torch.int64, device=device)
        dist.all_reduce(cap, op=dist.ReduceOp.MAX, group=group)
        self.capacity = max(int(cap.item()), 1)
        self.buf = symm_mem.empty(2 * self.capacity, dtype=dtype, device=device)
        self.buf.zero_()
        self.handle = symm_mem.rendezvous(self.buf, group)
        self.sends = []  # (owner, local gather positions, [view of the owner's buffer half 0, half 1])
        for o, idx in sends:
            off, length = int(table[o][rank]), int(table[o][world + rank])
            assert length == idx.numel(), "interface key lists disagree between sender and owner"
            remote = self.handle.get_buffer(o, (2 * self.capacity,), dtype)
            halves = [remote[h * self.capacity + off : h * self.capacity + off + length] for h in (0, 1)]
            self.sends.append((o, idx, halves))
        self.recvs = []  # (peer, local positions, [my buffer half 0, half 1])
        for p, idx in recvs:
            off = int(offsets[p])
            halves = [self.buf[h * self.capacity + off : h * self.capacity + off + idx.numel()] for h in (0, 1)]
            self.recvs.append((p, idx, halves))
        self.steps = 0
        self.bytes_per_exchange = sum(idx.numel() for _, idx, _ in self.sends) * self.buf.element_size()
        self.n_kernels = len(self.sends) + len(self.recvs)
        dist.barrier(group=group)  # every rank has mapped its peers before the first store

    def __call__(self, buffer: torch.Tensor):
        self.pack(buffer)
        self.gather_add(buffer)

    def pack(self, buffer: torch.Tensor, progress: Optional[torch.Tensor] = None, target: int = 0):
        """With `progress`, the pack kernels wait ON THE DEVICE for the assembly launch running beside
        them to finish its interface tiles (counter >= target) instead of for a stream event."""
        half = self.steps & 1
        for owner, idx, halves in self.sends:
            if self.steps >= 2:  # the owner has added what this half held two steps ago
                self.handle.wait_signal(owner, self.FREE + half, self.timeout_ms)
            if progress is None:
                self.ops.pack_into(halves[half], buffer, idx)
            else:
                from . import ops

                ops.pack_after_raw(halves[half], buffer, idx, progress, target)
            self.handle.put_signal(owner, self.DATA + half, self.timeout_ms)

    def wait_local(self, buffer: torch.Tensor, progress: torch.Tensor, target: int):
        """Order this stream after the interface tiles of the assembly launch running beside it, on a rank
        that only RECEIVES (a rank that sends is already ordered by its pack kernels, which wait for the
        same counter): without it the owner's add could race with its own tiles' plain stores."""
        if self.sends or not self.recvs:
            return
        from . import ops

        if getattr(self, "_wait_scratch", None) is None:
            self._wait_scratch = torch.zeros(1, dtype=buffer.dtype, device=buffer.device)
            self._wait_index = torch.zeros(1, dtype=torch.int32, device=buffer.device)
        ops.pack_after_raw(self._wait_scratch, buffer, self._wait_index, progress, target)

    def gather_add(self, buffer: torch.Tensor):
        half = self.steps & 1
        for peer, idx, halves in self.recvs:  # ascending peer order -> bitwise reproducible sums
            self.handle.wait_signal(peer, self.DATA + half, self.timeout_ms)
            self.ops.unpack_add(buffer, idx, halves[half])
            self.handle.put_signal(peer, self.FREE + half, self.timeout_ms)
        self.steps += 1


class PartitionedAssembly:
    """Element-partitioned assembly of ANY planar P1 triangle mesh: this rank holds a slice of the global
    element list (`conn_global`, global vertex ids), assembles it with the single-GPU kernels into a local
    CSR system and exchanges the interface rows with their owners (SURVEY.md 8(e)).

    `step()` is one persistent launch that walks the tiles holding interface rows first; the interface
    exchange (pack into the owner's peer buffer -> signal -> add) runs on a side stream while the same
    launch continues with the interior tiles.  With the collective transport (`TFEM_EXCHANGE=nccl`, gloo
    tests) the interface and interior tiles are two launches and the exchange sits between them.

    `vertices` is the global (n_global, 2) coordinate array or a callable `ids -> (len(ids), 2)`; only the
    vertices this rank's elements touch are ever looked at (ghost columns carry no geometry)."""

    def __init__(self, vertices, conn_global, n_global, rank, world, device, quad_order=3, rows_per_tile=336, group=None,
                 exchange_ops=None, markers=None):
        import numpy as np

        from . import ElementTri, MeshTri, forms

        conn_global = torch.as_tensor(conn_global).to(device=device, dtype=torch.int64)
        self.plan = InterfacePlan(conn_global, n_global, rank, world, group)
        local_ids = self.plan.local_to_global.cpu().numpy()
        touched = np.zeros(local_ids.shape[0], dtype=bool)
        touched[np.unique(self.plan.dof_conn.cpu().numpy())] = True
        coords = np.zeros((local_ids.shape[0], 2))
        coords[touched] = vertices(local_ids[touched]) if callable(vertices) else np.asarray(vertices)[local_ids[touched]]
        vertex_markers = np.zeros((local_ids.shape[0], 1), dtype=np.int32)
        if markers is not None:
            vertex_markers[touched] = np.asarray(markers).reshape(-1, 1)[local_ids[touched]]
        self.mesh_dict = {"vertices": coords, "triangles": self.plan.dof_conn.cpu().numpy().astype(np.int32), "vertex_markers": vertex_markers}
        self.local_to_global = self.plan.local_to_global
        with torch.device(device):
            self.basis = _basis_for(MeshTri(self.mesh_dict), ElementTri(1, quad_order))
        self.basis._pattern = csr_mod.build_pattern(self.basis._dof_conn_flat(), self.plan.n_local, self.plan.extra_keys)
        self.plan.bind(self.basis.pattern)
        self.exchange = InterfaceExchange(self.plan, exchange_ops)

        # one buffer for [values | load]; interface tiles and interior tiles as two sub-plans
        pat = self.basis.pattern
        self.quad_order = quad_order
        self.buffer = torch.empty(pat.nnz + pat.n_dof, dtype=self.basis.dtype, device=device)
        self.values, self.load = self.buffer[: pat.nnz], self.buffer[pat.nnz :]
        self.fused_exchange = self._make_exchange(pat.nnz, device, exchange_ops)
        full = self.basis.tile_plan(rows_per_tile)
        interface_local = torch.searchsorted(self.plan.local_to_global, self.plan.interface_global)
        is_interface_tile = torch.zeros(full.n_tiles, dtype=torch.bool, device=device)
        is_interface_tile[full.tile_of_row[interface_local]] = True
        # inside each group keep the plan's own order (congruent tiles adjacent: a CTA rarely changes template)
        order = full.default_order.long()
        self.interface_tiles = full.subset(order[is_interface_tile[order]])
        # the interior launch leaves some CTA slots free so the exchange kernels can run beside it
        reserve = int(os.environ.get("TFEM_RESERVE_CTAS", "8"))
        self.interior_tiles = full.subset(order[~is_interface_tile[order]], reserve_ctas=reserve)
        self.full_plan = full
        # one launch, interface tiles first, counted on a device counter the pack kernels wait for
        self.progress = torch.zeros(1, dtype=torch.int32, device=device)
        ids = torch.cat([self.interface_tiles.tile_list, self.interior_tiles.tile_list])
        self.n_interface_tiles = int(self.interface_tiles.tile_list.numel())
        self.ordered_tiles = full.subset(ids, reserve_ctas=reserve, n_progress_tiles=self.n_interface_tiles, progress=self.progress)
        self.progress_target = 0
        self.source = forms.SinSinSource()
        self.side_stream = torch.cuda.Stream(device=device) if torch.device(device).type == "cuda" else None
        self.single_launch = isinstance(self.fused_exchange, PeerExchange) and os.environ.get("TFEM_SINGLE_LAUNCH", "1") == "1"
        self._debug_no_exchange = os.environ.get("TFEM_DEBUG_NO_EXCHANGE", "0") == "1"
        self._previous_step = torch.cuda.Event() if self.side_stream is not None else None
        if self._previous_step is not None:
            self._previous_step.record(torch.cuda.current_stream())
        # ranks leave set-up together: the first step's device-side waits (bounded) then only see kernel-scale skew
        dist.barrier(group=self.plan.group)

    @classmethod
    def from_mesh(cls, mesh_dict, rank, world, device, **kwargs):
        """Strong scaling: rank `rank` takes the `rank`-th of `world` contiguous ranges of the mesh's element list."""
        import numpy as np

        triangles = np.asarray(mesh_dict["triangles"])
        n_el = triangles.shape[0]
        lo, hi = (n_el * rank) // world, (n_el * (rank + 1)) // world
        return cls(np.asarray(mesh_dict["vertices"]), triangles[lo:hi].astype(np.int64), int(np.asarray(mesh_dict["vertices"]).shape[0]),
                   rank, world, device, markers=mesh_dict.get("vertex_markers"), **kwargs)

    def _make_exchange(self, nnz, device, exchange_ops):
        """Peer-memory stores + signals on NVLink when the ranks are CUDA peers (TFEM_EXCHANGE=peer, the
        default with NCCL), else one all-gather (TFEM_EXCHANGE=nccl; gloo in the CPU tests)."""
        kind = os.environ.get("TFEM_EXCHANGE", "peer" if dist.get_backend(self.plan.group) == "nccl" else "nccl")
        if kind == "peer":
            try:
                return PeerExchange(self.plan, nnz, self.basis.dtype, device, exchange_ops)
            except Exception as error:  # no P2P mapping between these devices: say so, use the collective
                import sys

                print(f"[tfem] peer-memory exchange unavailable ({error!r}); using all_gather", file=sys.stderr)
        return FusedExchange(self.plan, nnz, self.basis.dtype, device, exchange_ops)

    def _launch(self, plan, alpha, beta, coords=None, buffer=None):
        from . import ops

        nnz = self.basis.pattern.nnz
        buffer = self.buffer if buffer is None else buffer
        ops.assemble_csr_tiled(plan.c_struct(), self.basis._layout.coords if coords is None else coords, self.quad_order,
                               alpha, beta, self.source.kind, self.source.params, buffer[:nnz], buffer[nnz:])

    def _single_launch_step(self, main, alpha, beta, coords, buffer, captured: bool):
        """ONE persistent launch walks the interface tiles first and counts them on a device counter; the pack
        kernels on the side stream wait for that counter, store over NVLink into the owners' buffers and signal,
        while the same launch goes on with the interior tiles.  `captured`: the call is being recorded into a CUDA
        graph."""
        # the counter restarts every step (the previous step's waiters are done: the calling stream has waited for
        # them), so eager steps and graph replays can be mixed and every replay waits for the same target
        target = self.n_interface_tiles * self.ordered_tiles.consumer_warps
        self.progress.zero_()
        # everything the calling stream has waited for so far (the previous step, and in the host pipeline
        # the copies that free `coords` / `buffer`) also gates the side stream
        entered = torch.cuda.Event()
        entered.record(main)
        self._launch(self.ordered_tiles, alpha, beta, coords, buffer)
        with torch.cuda.stream(self.side_stream):
            if not captured:
                self.side_stream.wait_event(self._previous_step)  # the buffer's previous contents are final
            self.side_stream.wait_event(entered)
            self.fused_exchange.pack(buffer, self.progress, target)
            self.fused_exchange.wait_local(buffer, self.progress, target)
            self.fused_exchange.gather_add(buffer)
            finished = torch.cuda.Event()
            finished.record(self.side_stream)
        main.wait_event(finished)
        if not captured:
            self._previous_step.record(main)

    def capture(self, alpha: float = 1.0, beta: float = 1.0) -> bool:
        """Record `step()` (assembly launch + side-stream exchange with its NVLink signals) into two CUDA graphs, one
        per receive-buffer half; `replay()` then costs one graph launch on the host instead of ~15 enqueues, which
        is what bounds a step once the per-rank work drops below ~90 us (strong scaling).  Returns False (and
        leaves `replay` = `step`) where the step cannot be captured."""
        self._graphs = None
        if not self.single_launch or self.side_stream is None or os.environ.get("TFEM_STEP_GRAPH", "1") != "1":
            return False
        exchange = self.fused_exchange
        while exchange.steps < 2 or exchange.steps & 1:  # past the start-up steps, next step on half 0
            self.step(alpha, beta)
        torch.cuda.synchronize()
        dist.barrier(group=self.plan.group)
        stream = torch.cuda.Stream(device=self.buffer.device)
        graphs = []
        try:
            from . import _lib

            for parity in (0, 1):
                assert exchange.steps & 1 == parity
                launches_before = sum(_lib.LAUNCHES.values())
                graph = torch.cuda.CUDAGraph()
                stream.wait_stream(torch.cuda.current_stream())
                with torch.cuda.graph(graph, stream=stream, capture_error_mode="thread_local"):
                    self._single_launch_step(torch.cuda.current_stream(), alpha, beta, None, self.buffer, captured=True)
                graphs.append(graph)
                self._graph_kernels = sum(_lib.LAUNCHES.values()) - launches_before  # our kernels inside one replay
                graph.replay()  # the recorded step has not run yet: run it, every rank the same parity
                torch.cuda.synchronize()
        except Exception as error:  # noqa: BLE001 - reported; the eager step keeps working
            import sys

            print(f"[tfem] step graph capture unavailable ({error!r}); using eager launches", file=sys.stderr)
            return False
        self._graphs = graphs
        self._graph_parity = exchange.steps & 1
        return True

    def replay(self):
        """One distributed assembly through the captured graphs (after `capture()`), else a plain `step()`."""
        if getattr(self, "_graphs", None) is None:
            return self.step()
        from . import _lib

        self._graphs[self._graph_parity].replay()
        self._graph_parity ^= 1
        self.fused_exchange.steps += 1
        _lib.LAUNCHES["graph_replay"] = _lib.LAUNCHES.get("graph_replay", 0) + self._graph_kernels

    def step(self, alpha: float = 1.0, beta: float = 1.0, coords: Optional[torch.Tensor] = None,
             buffer: Optional[torch.Tensor] = None):
        """One distributed assembly (owned rows complete) into `self.values` / `self.load`, or into
        `buffer` = `[values | load]` from the vertex coordinates `coords` when given (host pipeline)."""
        main = torch.cuda.current_stream()
        buffer = self.buffer if buffer is None else buffer
        if self._debug_no_exchange:  # profiling aid: the assembly launch alone (results incomplete on interface rows)
            self._launch(self.ordered_tiles, alpha, beta, coords, buffer)
            return
        if self.single_launch:
            self._single_launch_step(main, alpha, beta, coords, buffer, captured=False)
            return
        self._launch(self.interface_tiles, alpha, beta, coords, buffer)
        ready = torch.cuda.Event()
        ready.record(main)
        # enqueue the long interior launch BEFORE the exchange so the GPU is busy while the host issues
        # the pack / exchange / add sequence on the side stream
        self._launch(self.interior_tiles, alpha, beta, coords, buffer)
        with torch.cuda.stream(self.side_stream):
            self.side_stream.wait_event(ready)
            self.fused_exchange(buffer)
            finished = torch.cuda.Event()
            finished.record(self.side_stream)
        main.wait_event(finished)


class StripAssembly(PartitionedAssembly):
    """Weak-scaling driver of bench.py: every rank owns a 2*nx*ny-element strip of a mesh `world` times taller."""

    def __init__(self, nx, ny, rank, world, device, quad_order=3, rows_per_tile=336, group=None, exchange_ops=None):
        import numpy as np

        mesh, offset, n_global = strip_mesh(nx, ny, rank, world)
        strip_vertices = mesh["vertices"]

        def vertices(ids):  # global ids of this strip are local ids plus a constant
            return strip_vertices[ids - offset]

        super().__init__(vertices, mesh["triangles"].astype(np.int64) + offset, n_global, rank, world, device, quad_order, rows_per_tile,
                         group, exchange_ops)
        # strips are contiguous ranges of global ids, so local ids are global ids minus a constant
        # and ghosts (the vertex row above the strip) sort to the end: local numbering is unchanged
        assert torch.equal(self.plan.dof_conn.cpu(), torch.from_numpy(mesh["triangles"]).to(torch.int32))


class StripHostPipeline:
    """`StripAssembly.step` fed from / drained to pinned HOST memory with `depth` steps in flight: the
    host->device copy of step i+1, the distributed assembly of step i (launch + interface exchange) and
    the device->host copy of step i-1 overlap on three streams (see basis.HostPipeline for one GPU)."""

    def __init__(self, assembler: PartitionedAssembly, depth: int = 2):
        self.assembler, self.depth = assembler, max(int(depth), 1)
        coords = assembler.basis._layout.coords
        self.coords = [torch.empty_like(coords) for _ in range(self.depth)]
        self.buffers = [torch.empty_like(assembler.buffer) for _ in range(self.depth)]
        device = coords.device
        self.copy_in, self.compute, self.copy_out = (torch.cuda.Stream(device=device) for _ in range(3))
        self.in_done = [torch.cuda.Event() for _ in range(self.depth)]
        self.compute_done = [torch.cuda.Event() for _ in range(self.depth)]
        self.out_done = [torch.cuda.Event() for _ in range(self.depth)]
        self.submitted = 0
        self.nnz = assembler.basis.pattern.nnz

    def step(self, coords_host: torch.Tensor, values_host: torch.Tensor, load_host: torch.Tensor, alpha: float = 1.0, beta: float = 1.0):
        k = self.submitted % self.depth
        recycled = self.submitted >= self.depth
        with torch.cuda.stream(self.copy_in):
            if recycled:
                self.copy_in.wait_event(self.compute_done[k])
            self.coords[k].copy_(coords_host.reshape(self.coords[k].shape), non_blocking=True)
            self.in_done[k].record(self.copy_in)
        with torch.cuda.stream(self.compute):
            self.compute.wait_event(self.in_done[k])
            if recycled:
                self.compute.wait_event(self.out_done[k])
            self.assembler.step(alpha, beta, self.coords[k], self.buffers[k])
            self.compute_done[k].record(self.compute)
        with torch.cuda.stream(self.copy_out):
            self.copy_out.wait_event(self.compute_done[k])
            values_host.copy_(self.buffers[k][: self.nnz], non_blocking=True)
            load_host.copy_(self.buffers[k][self.nnz :].reshape(load_host.shape), non_blocking=True)
            self.out_done[k].record(self.copy_out)
        self.submitted += 1

    def synchronize(self):
        for stream in (self.copy_in, self.compute, self.copy_out):
            stream.synchronize()


def _basis_for(mesh, element):
    from . import Basis

    return Basis(mesh, element)


class PartitionedFractureAssembly:
    """Element-partitioned assembly of a FRACTURE NETWORK (SURVEY.md 8(e), BASELINE config 5): rank `rank` takes the
    `rank`-th of `world` contiguous ranges of the flattened element list of `FractureBasis` -- the list behind
    `global_triangles` (basis/fracture_basis.py:65-69), so a cut may fall inside a fracture or between two -- and
    assembles it in one launch of the tiled kernel with the fractures' metrics
    (`tfem_tri_p1_assemble_csr_ex`); rows shared with other ranks (cut lines, trace vertices) are summed at
    their owner (`InterfacePlan` / `InterfaceExchange`), in fixed rank order.

    `basis` is the whole network's `FractureBasis` on this rank's device: only its index structures and the vertex
    coordinates are used (set-up); the per-step work touches this rank's elements alone."""

    def __init__(self, basis, rank: int, world: int, group=None, rows_per_tile: int = 336, exchange_ops: Optional[ExchangeOps] = None):
        import math

        lay = basis._layout
        if lay.frac is None:
            raise ValueError("PartitionedFractureAssembly needs a FractureBasis; planar meshes use PartitionedAssembly")
        device = lay.coords.device
        n_el, per_mesh = lay.n_total, lay.n_el_per_mesh
        self.lo, self.hi = (n_el * rank) // world, (n_el * (rank + 1)) // world
        offsets = (torch.arange(n_el, device=device) // per_mesh) * lay.n_vert_per_mesh
        geom_conn = (lay.conn.long() + offsets[:, None])[self.lo : self.hi]
        dof_global = basis._dof_conn_flat().long()[self.lo : self.hi]
        self.basis, self.rank, self.world = basis, rank, world
        self.plan = InterfacePlan(dof_global, basis.n_dof_flat, rank, world, group)
        self.pattern = csr_mod.build_pattern(self.plan.dof_conn, self.plan.n_local, self.plan.extra_keys)
        self.plan.bind(self.pattern)
        # rows are clustered fracture by fracture (all fractures share one local 2-D frame)
        points = torch.zeros((self.plan.n_local, 2), dtype=lay.coords.dtype, device=device)
        local = lay.coords[geom_conn.reshape(-1)].clone()
        span = float(lay.coords[:, 0].max() - lay.coords[:, 0].min())  # side by side, no gaps: the blocks stay full
        fracture_of = torch.div(torch.arange(self.lo, self.hi, device=device), per_mesh, rounding_mode="floor")
        local[:, 0] += span * fracture_of.repeat_interleave(3).to(local.dtype)
        points[self.plan.dof_conn.reshape(-1).long()] = local
        self.tile_plan = csr_mod.build_tile_plan(geom_conn, self.plan.dof_conn, self.pattern, points, rows_per_tile, "block", elem_ids=True)
        # the kernel finds an element's fracture as (local element id) / n_el_per_mesh: give it a metric table in units of
        # g = gcd(elements per fracture, first element of the range), in which the range's fracture boundaries are whole rows
        g = math.gcd(per_mesh, self.lo) if self.lo else per_mesh
        rows = (self.hi - self.lo + g - 1) // g
        fracture_of_row = torch.div(self.lo // g + torch.arange(rows, device=device), per_mesh // g, rounding_mode="floor")
        self.metric = basis._fracture_metric()[fracture_of_row.clamp_max(n_el // per_mesh - 1)].contiguous()
        self.metric_unit = g
        self.coords = lay.coords
        self.quad_order = basis._element.integration_order
        self.exchange = InterfaceExchange(self.plan, exchange_ops)
        self.values = torch.empty(self.pattern.nnz, dtype=basis.dtype, device=device)
        self.load = torch.empty(self.pattern.n_dof, dtype=basis.dtype, device=device)

    def step(self, bilinear=None, source=None):
        """One distributed assembly: this rank's elements into `self.values` / `self.load` (local CSR of
        `self.pattern`), then the interface exchange; owned rows (`self.plan.owned_rows`) are complete afterwards."""
        from . import forms, ops

        src = forms.as_source(source)
        want_mat, want_vec = bilinear is not None, source is not None
        if want_mat and bilinear.has_field:
            raise NotImplementedError("the distributed assembly runs the tiled kernel, which takes constant coefficients only")
        f_q = None
        if want_vec and src.kind == ops.SRC_SAMPLED:
            f_q = self.basis._sampled_source(src)[self.lo : self.hi].contiguous()
        alpha, beta = (bilinear.alpha, bilinear.beta) if want_mat else (0.0, 0.0)
        ops.assemble_csr_tiled(self.tile_plan, self.coords, self.quad_order, alpha, beta, src.kind if want_vec else 0, src.params,
                               self.values if want_mat else None, self.load if want_vec else None, f_q, self.metric_unit, self.metric)
        self.exchange(self.values if want_mat else None, self.load if want_vec else None)
        return (self.values if want_mat else None), (self.load if want_vec else None)
