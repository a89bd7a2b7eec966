"""Spatial domain decomposition of one large periodic cell across ranks (BASELINE.json config 4).

Nothing in the reference corresponds to this (nn/gradient.py:26 "TODO: current implementation cannot be used with
spatial decomposition").  Scheme (SURVEY.md §7 "scheme B"): every rank owns the atoms of one box of a
(gx, gy, gz) grid in fractional space and imports one r_c-wide ghost shell.  Every directed edge i→j and every
triplet is owned by its source / centre atom, so edge features never cross ranks; only node features of ghost
atoms do:

  per step     ghost positions are part of the local structure (owner position + image shift)
  per block    forward halo:  x[ghost] <- x[owner]            (N_ghost x F floats, after every M3GNetConv but the last)
               reverse halo:  dE/dx[owner] += dE/dx[ghost]    (in the backward pass)
  per step     reverse halo of dE/dpos, then forces of the owned atoms; energies are summed with all_reduce.

The exchange is an ``all_to_all_single`` over NCCL (NVLink / NVSwitch); messages are small (≤ ~1 MB), so the cost
is latency, not bandwidth.  The same plan drives an in-process emulation of all ranks on one GPU
(``evaluate_emulated``), which is what the single-GPU test-suite checks against the undecomposed model.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from torch_m3gnet_b200.data import MaterialGraphKey as K
from torch_m3gnet_b200.data.material_graph import Batch
from torch_m3gnet_b200.nn.conv import M3GNetConv


class DomainPlan:
    """Host-side partition of one structure: owners, ghosts (atom, image) and the send/recv lists of every rank."""

    def __init__(self, lattice: np.ndarray, cart: np.ndarray, atomic_numbers: np.ndarray, grid: Sequence[int],
                 cutoff: float):
        lattice = np.asarray(lattice, dtype=np.float64).reshape(3, 3)
        cart = np.asarray(cart, dtype=np.float64).reshape(-1, 3)
        self.lattice, self.cart, self.z = lattice, cart, np.asarray(atomic_numbers, dtype=np.int64)
        self.grid = tuple(int(g) for g in grid)
        self.world = int(np.prod(self.grid))
        self.cutoff = float(cutoff)
        inv = np.linalg.inv(lattice)
        heights = 1.0 / np.linalg.norm(inv, axis=0)
        margin = (cutoff + 1e-6) / heights  # ghost-shell width in fractional units
        for k in range(3):
            if 1.0 / self.grid[k] < margin[k] and self.grid[k] > 1:
                raise ValueError(f"domain width along axis {k} is smaller than the cutoff")
            if margin[k] >= 1.0:
                raise ValueError("cell is thinner than the cutoff: use structure sharding, not domain decomposition")
        frac = cart @ inv
        wrap = np.floor(frac)
        f0 = frac - wrap  # in [0,1)
        cell = np.minimum((f0 * np.array(self.grid)).astype(np.int64), np.array(self.grid) - 1)
        owner = (cell[:, 0] * self.grid[1] + cell[:, 1]) * self.grid[2] + cell[:, 2]
        self.owner = owner
        self.owned: List[np.ndarray] = [np.nonzero(owner == r)[0] for r in range(self.world)]
        local_of = np.empty(len(cart), dtype=np.int64)
        for r in range(self.world):
            local_of[self.owned[r]] = np.arange(len(self.owned[r]))
        shifts = np.stack(np.meshgrid(*[np.arange(-1, 2)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
        # ghosts[r] = list of (atom, image) ordered by (owner rank, position in the owner's send list)
        self.ghost_atom: List[np.ndarray] = []
        self.ghost_image: List[np.ndarray] = []
        self.recv_counts = np.zeros((self.world, self.world), dtype=np.int64)  # [r][q]: r receives from q
        self.send_index: List[List[np.ndarray]] = [[None] * self.world for _ in range(self.world)]  # [q][r]
        for r in range(self.world):
            c = np.array([r // (self.grid[1] * self.grid[2]), (r // self.grid[2]) % self.grid[1], r % self.grid[2]])
            lo = c / np.array(self.grid) - margin
            hi = (c + 1) / np.array(self.grid) + margin
            atoms, images = [], []
            for s in shifts:
                fs = f0 + s  # position of the image in fractional units (wrapped coordinates)
                inside = np.all((fs >= lo) & (fs < hi), axis=1)
                if not s.any():
                    inside &= owner != r
                idx = np.nonzero(inside)[0]
                if idx.size:
                    atoms.append(idx)
                    # image relative to the UNWRAPPED input coordinate of the atom
                    images.append(np.broadcast_to(s, (idx.size, 3)) - wrap[idx].astype(np.int64))
            atoms = np.concatenate(atoms) if atoms else np.zeros(0, np.int64)
            images = np.concatenate(images) if images else np.zeros((0, 3), np.int64)
            order = np.lexsort((images[:, 2], images[:, 1], images[:, 0], atoms, owner[atoms])) if atoms.size else \
                np.zeros(0, np.int64)
            atoms, images = atoms[order], images[order]
            self.ghost_atom.append(atoms)
            self.ghost_image.append(images)
            for q in range(self.world):
                sel = owner[atoms] == q
                self.recv_counts[r, q] = int(sel.sum())
                self.send_index[q][r] = local_of[atoms[sel]]
        self.wrap = wrap.astype(np.int64)

    def local_arrays(self, r: int) -> Tuple[np.ndarray, np.ndarray, int]:
        """Positions (owned first, unwrapped-in-place; ghosts = atom + image·lattice) and atomic numbers of rank r."""
        own = self.owned[r]
        # owned atoms are used at their wrapped position so that the local cloud is compact
        own_pos = self.cart[own] - self.wrap[own] @ self.lattice
        g_atoms, g_img = self.ghost_atom[r], self.ghost_image[r]
        ghost_pos = self.cart[g_atoms] + g_img @ self.lattice
        pos = np.concatenate([own_pos, ghost_pos]) if len(g_atoms) else own_pos
        z = np.concatenate([self.z[own], self.z[g_atoms]]) if len(g_atoms) else self.z[own]
        return pos, z, len(own)

    def send_concat(self, q: int) -> Tuple[np.ndarray, List[int]]:
        """Rows rank q packs (ordered by destination rank) and the per-destination counts."""
        parts = [self.send_index[q][r] for r in range(self.world)]
        counts = [len(p) for p in parts]
        return (np.concatenate(parts) if sum(counts) else np.zeros(0, np.int64)), counts


class DomainBatch:
    """The local graph of one rank: owned + ghost atoms in one non-periodic structure, edges of owned sources only."""

    def _exchange_fields(self, dev):
        plan, rank = self.plan, self.rank
        send, send_counts = plan.send_concat(rank)
        self.send_idx = torch.as_tensor(send, dtype=torch.long, device=dev)
        self.send_counts = [int(c) for c in send_counts]
        self.recv_counts = [int(c) for c in plan.recv_counts[rank]]
        self.global_owned = torch.as_tensor(plan.owned[rank], dtype=torch.long, device=dev)

    @classmethod
    def exchange_only(cls, plan: DomainPlan, rank: int, device="cpu") -> "DomainBatch":
        """Only the halo-exchange bookkeeping (no graph): used by the host-side (gloo) tests of the exchange."""
        self = object.__new__(cls)
        self.plan, self.rank = plan, rank
        self.n_own = len(plan.owned[rank])
        self.n_local = self.n_own + len(plan.ghost_atom[rank])
        self.graph = None
        self._exchange_fields(torch.device(device))
        return self

    def __init__(self, plan: DomainPlan, rank: int, cutoff: float, threebody_cutoff: float, device):
        self.plan, self.rank = plan, rank
        pos, z, n_own = plan.local_arrays(rank)
        self.n_own, self.n_local = n_own, len(pos)
        span = pos.max(axis=0) - pos.min(axis=0) if len(pos) else np.ones(3)
        box = np.diag(span + 4.0 * cutoff + 1.0)  # no periodic image of the cloud lies within the cutoff
        full = Batch.from_arrays(box[None], pos, z, [len(pos)], cutoff, threebody_cutoff, device=device)
        fp = full._plan
        e_keep = int(fp.edge_ptr[n_own].item())
        t_keep = int(fp.tri_ptr[e_keep].item()) if e_keep > 0 else 0
        n_ghost = self.n_local - n_own
        dev = full[K.POS].device
        g = Batch(pos=full[K.POS], atom_types=full[K.ATOM_TYPES], num_triplet_i=full[K.NUM_TRIPLET_I],
                  edge_index=full[K.EDGE_INDEX][:, :e_keep].contiguous(),
                  edge_cell_shift=full[K.EDGE_CELL_SHIFT][:e_keep].contiguous(),
                  num_triplet_ij=full[K.NUM_TRIPLET_IJ][:e_keep].contiguous(),
                  triplet_edge_index=full[K.TRIPLET_EDGE_INDEX][:, :t_keep].contiguous(),
                  lattice=torch.stack([full[K.LATTICE][0], full[K.LATTICE][0]]))
        # two "structures": 0 = owned atoms (energy counted), 1 = ghosts (energy discarded)
        g[K.BATCH] = torch.cat([torch.zeros(n_own, dtype=torch.long, device=dev),
                                torch.ones(n_ghost, dtype=torch.long, device=dev)])
        self.graph = g
        self._exchange_fields(dev)


# ----------------------------------------------------------------------------------------------------------------
# halo exchange as autograd functions
# ----------------------------------------------------------------------------------------------------------------
class DistHaloFn(torch.autograd.Function):
    """One rank's view: ghost rows of ``x`` are replaced by the owners' rows (all_to_all_single); the backward adds
    the ghost-row gradients into the owners' rows."""

    @staticmethod
    def forward(ctx, x, dbatch: DomainBatch, group):
        import torch.distributed as dist

        send = x.index_select(0, dbatch.send_idx).contiguous()
        recv = x.new_empty((sum(dbatch.recv_counts),) + tuple(x.shape[1:]))
        dist.all_to_all_single(recv, send, dbatch.recv_counts, dbatch.send_counts, group=group)
        out = x.clone()
        out[dbatch.n_own:] = recv
        ctx.dbatch, ctx.group = dbatch, group
        return out

    @staticmethod
    def backward(ctx, g):
        import torch.distributed as dist

        d = ctx.dbatch
        g_ghost = g[d.n_own:].contiguous()
        back = g.new_empty((sum(d.send_counts),) + tuple(g.shape[1:]))
        dist.all_to_all_single(back, g_ghost, d.send_counts, d.recv_counts, group=ctx.group)
        g_in = g.clone()
        g_in[d.n_own:] = 0
        g_in.index_add_(0, d.send_idx, back)
        return g_in, None, None


class EmulatedHaloFn(torch.autograd.Function):
    """All ranks in one process (single-GPU emulation of the exchange; same plan, same ordering)."""

    @staticmethod
    def forward(ctx, dbatches, *xs):
        outs = [x.clone() for x in xs]
        world = len(xs)
        for r in range(world):
            off = dbatches[r].n_own
            for q in range(world):
                cnt = dbatches[r].recv_counts[q]
                if cnt:
                    s0 = sum(dbatches[q].send_counts[:r])
                    outs[r][off:off + cnt] = xs[q].index_select(0, dbatches[q].send_idx[s0:s0 + cnt])
                off += cnt
        ctx.dbatches = dbatches
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gs):
        dbatches = ctx.dbatches
        world = len(gs)
        g_in = []
        for r in range(world):
            t = gs[r].clone()
            t[dbatches[r].n_own:] = 0
            g_in.append(t)
        for r in range(world):
            off = dbatches[r].n_own
            for q in range(world):
                cnt = dbatches[r].recv_counts[q]
                if cnt:
                    s0 = sum(dbatches[q].send_counts[:r])
                    g_in[q].index_add_(0, dbatches[q].send_idx[s0:s0 + cnt], gs[r][off:off + cnt])
                off += cnt
        return (None,) + tuple(g_in)


def _no_cell_stress(model):
    if getattr(model, "compute_stress", False):
        raise NotImplementedError("the cell stress (compute_stress) is not implemented for domain-decomposed cells: "
                                  "ghost bonds and the cross-rank reduction are not handled")


def _modules_of(model):
    _no_cell_stress(model)
    seq = model.model if hasattr(model, "model") else model
    mods = list(seq)
    last_conv = max(i for i, m in enumerate(mods) if isinstance(m, M3GNetConv))
    return mods, last_conv


def evaluate_distributed(model, dbatch: DomainBatch, group=None) -> Dict[str, torch.Tensor]:
    """Energy (global, all-reduced) and forces of the atoms this rank owns.  One process per GPU."""
    import torch.distributed as dist

    mods, last_conv = _modules_of(model)
    graph = dbatch.graph
    pos = graph[K.POS]
    pos.requires_grad_(True)
    for i, m in enumerate(mods):
        graph = m(graph)
        if isinstance(m, M3GNetConv) and i != last_conv:
            graph[K.NODE_FEATURES] = DistHaloFn.apply(graph[K.NODE_FEATURES], dbatch, group)
    energy = graph[K.TOTAL_ENERGY]
    weight = getattr(dbatch, "_energy_weight", None)
    if weight is None:  # built once: a host -> device copy would not be capturable in a CUDA graph
        weight = dbatch._energy_weight = torch.tensor([1.0, 0.0], device=energy.device)
    (g_pos,) = torch.autograd.grad(energy, pos, grad_outputs=weight)
    pos.requires_grad_(False)
    # reverse halo of dE/dpos: ghost gradients go home
    back = g_pos.new_empty((sum(dbatch.send_counts), 3))
    dist.all_to_all_single(back, g_pos[dbatch.n_own:].contiguous(), dbatch.send_counts, dbatch.recv_counts, group=group)
    g_own = g_pos[:dbatch.n_own].clone()
    g_own.index_add_(0, dbatch.send_idx, back)
    e_total = energy[0:1].detach().clone()
    dist.all_reduce(e_total, group=group)
    graph._private.clear()
    return {"total_energy": e_total, "forces": -g_own, "owned": dbatch.global_owned,
            "local_energy": energy[0:1].detach()}


def evaluate_emulated(model, dbatches: List[DomainBatch]) -> Dict[str, torch.Tensor]:
    """All ranks of a plan evaluated in lockstep on one GPU; returns the global energy and forces in atom order."""
    mods, last_conv = _modules_of(model)
    graphs = [d.graph for d in dbatches]
    for g in graphs:
        g[K.POS].requires_grad_(True)
    for i, m in enumerate(mods):
        graphs = [m(g) for g in graphs]
        if isinstance(m, M3GNetConv) and i != last_conv:
            xs = EmulatedHaloFn.apply(dbatches, *[g[K.NODE_FEATURES] for g in graphs])
            for g, x in zip(graphs, xs):
                g[K.NODE_FEATURES] = x
    energies = [g[K.TOTAL_ENERGY] for g in graphs]
    total = sum(e[0] for e in energies)
    grads = torch.autograd.grad(total, [g[K.POS] for g in graphs])
    n_atoms = len(dbatches[0].plan.cart)
    forces = torch.zeros((n_atoms, 3), dtype=torch.float32, device=grads[0].device)
    plan = dbatches[0].plan
    for r, (d, gp) in enumerate(zip(dbatches, grads)):
        graphs[r][K.POS].requires_grad_(False)
        forces.index_add_(0, d.global_owned, -gp[: d.n_own])
        if len(plan.ghost_atom[r]):
            ghost_global = torch.as_tensor(plan.ghost_atom[r], dtype=torch.long, device=gp.device)
            forces.index_add_(0, ghost_global, -gp[d.n_own:])
        graphs[r]._private.clear()
    return {"total_energy": total.detach().reshape(1), "forces": forces}



# ----------------------------------------------------------------------------------------------------------------
# the same evaluation on the whole-step executor (engine.py): no autograd, the halo exchanges sit between the phases
# ----------------------------------------------------------------------------------------------------------------
class DomainStep:
    """Energy + forces of one rank's sub-domain through ``m3g_step_run`` phases with the halo exchanges in between:

        prologue, TB(0), CONV(0)  | x halo |  TB(1), CONV(1)  | x halo | ... READOUT
        CONV_BWD(n-1), TB_BWD(n-1) | reverse x halo | CONV_BWD(n-2) ... TB_BWD(0), EPILOGUE | reverse pos halo | FORCES

    Per step: (n_blocks - 1) forward halos of x (N_ghost x 64 floats), as many reverse halos of dE/dx, one reverse halo
    of dE/dpos and one all_reduce of the energy; pack / unpack are ``m3g_rows_gather`` / ``m3g_rows_scatter_add``.
    The buffers are allocated once, so the whole step (kernels + NCCL exchanges) can be captured in a CUDA graph
    (``capture=True``) and replayed: one host launch per step instead of ~70, which is what a sub-domain of a few
    thousand atoms needs.  New positions go in through ``set_positions``."""

    def __init__(self, model, dbatch: DomainBatch, group=None, capture: bool = False, warmup: int = 2,
                 exchange: str = "nccl"):
        """exchange = "nccl": all_to_all_single per halo.  exchange = "p2p": every halo is ONE kernel that packs the rows
        and stores them straight into the peers' landing buffers over NVLink / NVSwitch (peer-mapped symmetric memory,
        ``m3g_rows_put``), ordered by a device-side barrier; no collective call is left in the step (the energy sum
        goes the same way), so a captured step holds kernels only."""
        import torch.distributed as dist

        from torch_m3gnet_b200 import engine as E
        from torch_m3gnet_b200.data.material_graph import get_plan

        _no_cell_stress(model)

        self.dist, self.E, self.group = dist, E, group
        self.model, self.dbatch = model, dbatch
        self.engine = model.step_engine()
        graph = dbatch.graph
        plan = get_plan(graph)
        if not self.engine.supports(graph, plan):
            raise RuntimeError("DomainStep needs the default model shape (whole-step executor); use "
                               "evaluate_distributed for other models")
        dev = graph[K.POS].device
        self.device = dev
        self.n = self.engine.n_blocks
        self.weight = torch.tensor([1.0, 0.0], device=dev)  # structure 0 = owned atoms, 1 = ghosts
        self.desc, self.keep = self.engine.prepare(graph, plan, g_total=self.weight)
        scratch, off = self.keep["scratch"], self.keep["off"]
        N = plan.N

        def view(name, rows, width):
            return scratch[off[name]: off[name] + rows * width].view(rows, width)

        self.x_next = [view(f"x{b + 1}", N, 64) for b in range(self.n - 1)]  # output of CONV(b), input of block b+1
        self.g_x = [view("g_x0", N, 64), view("g_x1", N, 64)]
        self.g_pos = view("g_pos", N, 3)
        self.n_own = dbatch.n_own
        self.send_idx = dbatch.send_idx.to(torch.int32).contiguous()
        self.n_send = int(self.send_idx.numel())
        self.send_counts, self.recv_counts = dbatch.send_counts, dbatch.recv_counts
        self.send64 = torch.empty((max(self.n_send, 1), 64), device=dev)
        self.send3 = torch.empty((max(self.n_send, 1), 3), device=dev)
        self.pos = self.keep["inputs"][0]          # the (contiguous, detached) position buffer the kernels read
        out = self.keep["out"]
        self.energy = torch.zeros(1, device=dev)
        self.forces_local = out[K.FORCES]
        self.local_energy = out[K.TOTAL_ENERGY]
        self.exchanges_per_step = 2 * (self.n - 1) + 2
        self.exchange = exchange
        if exchange == "p2p":
            self._setup_p2p()
        elif exchange != "nccl":
            raise ValueError("exchange must be 'nccl' or 'p2p'")
        self.graph = None
        if capture:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(max(warmup, 1)):
                    self._step()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            # thread_local: the NCCL watchdog thread keeps polling its events while this thread captures
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._step()
            self.graph = g

    # ---- peer-memory exchange ---------------------------------------------------------------------------------
    def _setup_p2p(self):
        import torch.distributed._symmetric_memory as symm_mem

        dist, dev, plan, me = self.dist, self.device, self.dbatch.plan, self.dbatch.rank
        world = plan.world
        rc = plan.recv_counts  # [r][q]: r receives from q  (= q sends to r)
        n_ghost = [int(rc[r].sum()) for r in range(world)]
        n_send = [int(rc[:, q].sum()) for q in range(world)]
        G, S, nx = max(max(n_ghost), 1), max(max(n_send), 1), self.n - 1
        # landing zones (floats), the same layout on every rank: one zone per exchange of the step, so that a zone is
        # only rewritten after every rank has passed the barriers of all later exchanges
        self.z_fwd = [k * G * 64 for k in range(nx)]
        self.z_rev = [nx * G * 64 + k * S * 64 for k in range(nx)]
        self.z_pos = nx * (G + S) * 64
        self.z_en = self.z_pos + ((3 * S + 3) // 4) * 4
        total = self.z_en + ((world + 3) // 4) * 4
        self.land = symm_mem.empty(total, dtype=torch.float32, device=dev)
        self.land.zero_()
        group = self.group if self.group is not None else dist.group.WORLD
        self.hdl = symm_mem.rendezvous(self.land, group)
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        i64 = dict(dtype=torch.int64, device=dev)
        # forward: my send rows are ordered by destination rank r; on r they land behind the rows of the owners q < me
        dest = np.repeat(np.arange(world), self.send_counts)
        pos_in_chunk = np.concatenate([np.arange(c) for c in self.send_counts]) if self.n_send else np.zeros(0, np.int64)
        land_row = np.array([int(rc[r, :me].sum()) for r in range(world)])[dest] + pos_in_chunk if self.n_send else dest
        base = np.array(ptrs, dtype=np.int64)[dest] if self.n_send else np.zeros(0, np.int64)
        self.addr_fwd = [torch.as_tensor(base + 4 * (z + land_row * 64), **i64) for z in self.z_fwd]
        # reverse: my ghost rows are ordered by owner rank q; on q they land behind the rows q sent to ranks r < me
        n_g = self.dbatch.n_local - self.n_own
        owner = np.repeat(np.arange(world), self.recv_counts)
        pos_g = np.concatenate([np.arange(c) for c in self.recv_counts]) if n_g else np.zeros(0, np.int64)
        back_row = np.array([int(rc[:me, q].sum()) for q in range(world)])[owner] + pos_g if n_g else owner
        gbase = np.array(ptrs, dtype=np.int64)[owner] if n_g else np.zeros(0, np.int64)
        self.addr_rev = [torch.as_tensor(gbase + 4 * (z + back_row * 64), **i64) for z in self.z_rev]
        self.addr_pos = torch.as_tensor(gbase + 4 * (self.z_pos + back_row * 3), **i64)
        self.addr_en = torch.as_tensor(np.array(ptrs, dtype=np.int64) + 4 * (self.z_en + me), **i64)
        self.zero_idx = torch.zeros(world, dtype=torch.int32, device=dev)
        self.n_ghost = n_g
        self._chan = 0
        dist.barrier(group=self.group)
        torch.cuda.synchronize(dev)

    def _barrier(self):
        # device-side barrier of the symmetric-memory handle (a kernel on this stream): the peers' stores issued
        # before their barrier are visible after ours
        self.hdl.barrier(channel=self._chan)
        self._chan = (self._chan + 1) % 8

    # ---- halo exchanges -------------------------------------------------------------------------------------
    def _halo_forward(self, x, k=0):
        from torch_m3gnet_b200._lib import call

        if self.exchange == "p2p":
            call("rows_put", x, self.send_idx, self.addr_fwd[k], self.n_send, 64)
            self._barrier()
            z = self.z_fwd[k]
            x[self.n_own:].copy_(self.land[z: z + self.n_ghost * 64].view(self.n_ghost, 64))
            return

        call("rows_gather", x, self.send_idx, self.n_send, 64, self.send64)
        self.dist.all_to_all_single(x[self.n_own:], self.send64[: self.n_send], self.recv_counts, self.send_counts,
                                    group=self.group)

    def _halo_reverse(self, g, send_buf, width, k=0):
        from torch_m3gnet_b200._lib import call

        if self.exchange == "p2p":
            addr, z = (self.addr_rev[k], self.z_rev[k]) if width == 64 else (self.addr_pos, self.z_pos)
            call("rows_put", g[self.n_own:], None, addr, self.n_ghost, width)
            self._barrier()
            g[self.n_own:].zero_()
            call("rows_scatter_add", self.land[z: z + self.n_send * width], self.send_idx, self.n_send, width, g)
            return

        self.dist.all_to_all_single(send_buf[: self.n_send], g[self.n_own:], self.send_counts, self.recv_counts,
                                    group=self.group)
        g[self.n_own:].zero_()
        call("rows_scatter_add", send_buf, self.send_idx, self.n_send, width, g)

    def _step(self):
        E, n, d, dev = self.E, self.n, self.desc, self.device
        run = self.engine.run_phases
        run(d, 0, E.phase_conv(0), dev)
        for b in range(1, n):
            self._halo_forward(self.x_next[b - 1], b - 1)
            run(d, E.phase_tb(b), E.phase_conv(b), dev)
        run(d, E.phase_readout(n), E.phase_readout(n), dev)
        for b in range(n - 1, -1, -1):
            if b < n - 1:
                self._halo_reverse(self.g_x[d.cur_x], self.send64, 64, b)
            run(d, E.phase_conv_bwd(n, b), E.phase_tb_bwd(n, b), dev)
        run(d, E.phase_epilogue(n), E.phase_epilogue(n), dev)
        self._halo_reverse(self.g_pos, self.send3, 3)
        run(d, E.phase_forces(n), E.phase_forces(n), dev)
        if self.exchange == "p2p":
            from torch_m3gnet_b200._lib import call

            world = len(self.send_counts)
            call("rows_put", self.local_energy, self.zero_idx, self.addr_en, world, 1)
            self._barrier()
            torch.sum(self.land[self.z_en: self.z_en + world], dim=0, keepdim=True, out=self.energy)
        else:
            self.energy.copy_(self.local_energy[0:1])
            self.dist.all_reduce(self.energy, group=self.group)

    def set_positions(self, pos_local: torch.Tensor):
        """New local coordinates (owned atoms first, then ghosts, as in ``DomainPlan.local_arrays``); the bond list of
        the sub-domain is kept (rebuild the DomainBatch when atoms have moved further than its skin allows)."""
        self.pos.copy_(pos_local)

    def __call__(self) -> Dict[str, torch.Tensor]:
        if self.graph is not None:
            self.graph.replay()
        else:
            self._step()
        return {"total_energy": self.energy, "forces": self.forces_local[: self.n_own], "owned": self.dbatch.global_owned,
                "local_energy": self.local_energy[0:1]}
