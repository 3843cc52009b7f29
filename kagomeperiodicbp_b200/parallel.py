"""Multi-GPU block BP: one process per GPU (torch.distributed; NCCL on the GPU box, gloo in the CPU tests).

Two shardings, both from SURVEY 8e:
  * independent unit cells (ensembles, field sweeps): every rank runs whole BP / ITE problems, no data-path collective;
    only scalars are gathered at the end  (``gather_scalars``).
  * block sides of ONE unit cell: the six outgoing messages of an iteration depend only on the previous iteration's six
    messages (src/algo/belief_propagation.py:149-155), so rank r computes the chains of the sides ``sides_of_rank(r)`` on its
    GPU and ONE all-gather per BP iteration publishes every rank's new messages (+ its overlap / truncation scalars) to all
    ranks.  ``ShardedSides`` keeps everything on the device: the side programs write their outputs into one block of their
    arena, the all-gather runs on views of those blocks (NCCL straight between the GPUs' HBM), and the next iteration's
    inputs are filled from the gathered buffer by one indexed device copy per local program.  The host only reads the six
    overlaps (the convergence test of the BP loop).  Payload: 6 x (2N-1) sites of [chi, D^2, chi] complex128 (x2 with damping:
    the undamped message is what the error is measured on, the damped one is what the next iteration consumes).
Inside a chain the swallow steps are strictly sequential: nothing else shards.
"""
from __future__ import annotations

import numpy as np

from . import belief_propagation as bp
from .lattice import BLOCK_SIDES_CCW, SIDE_OPPOSITE


def sides_of_rank(rank: int, world: int):
    """round-robin over the counter-clockwise side order: 2 ranks -> 3+3, 4 ranks -> 2+2+1+1, >= 6 ranks -> 1 each (rest idle)."""
    return [s for k, s in enumerate(BLOCK_SIDES_CCW) if k % world == rank]


class ShardedSides:
    """device-resident BP iterations of ONE unit cell with its six sides sharded over the ranks of the default process group.

    Layout of a rank's contribution to the all-gather (float64 words): for each of its sides, in order,
    [ out block of the side program (complex128, 2 words each) | the program's slot row ], padded to the widest rank.
    """

    def __init__(self, N: int, cell, messages: dict, config, rank: int, world: int, device: int = 0, group=None, engine_key="side"):
        import torch
        self.torch = torch
        self.N, self.cell, self.config, self.rank, self.world, self.group = N, cell, config, rank, world, group
        d, D = cell.A.shape[0], cell.A.shape[1]
        shapes = bp._msg_shapes(messages)
        self.damping = config.damping if config.damping else None
        self.comps = {s: bp.compile_side_program(N, d, D, s, config.trunc_dim, shapes, self.damping) for s in BLOCK_SIDES_CCW}
        self.mine = sides_of_rank(rank, world)
        # the messages LIVE in these engines' arenas between steps: nothing else may run programs on them meanwhile
        self.engs = {s: bp.get_engine((engine_key, s), device) for s in self.mine}
        self.n_slots = bp.N_SLOTS
        # words each side contributes, and where each side's block sits in the gathered buffer [world, width]
        self.words = {s: 2 * self.comps[s].out_elems + self.n_slots for s in BLOCK_SIDES_CCW}
        per_rank = [sum(self.words[s] for s in sides_of_rank(r, world)) for r in range(world)]
        self.width = max(per_rank)
        self.gather_bytes = self.width * 8 * world
        self.pos = {}
        for r in range(world):
            p = 0
            for s in sides_of_rank(r, world):
                self.pos[s] = r * self.width + p
                p += self.words[s]
        # load programs, upload the cell tensors and the starting messages once
        for s in self.mine:
            comp, eng = self.comps[s], self.engs[s]
            comp.load(eng, 1)
            eng.upload(0, comp.pack_inputs([bp._side_inputs(cell, messages, comp)]))
            eng.sync()
        import torch.distributed as dist
        self.on_cuda = dist.get_backend(group) == "nccl"
        self.stream = None
        if self.on_cuda:                  # ranks beyond the sixth own no side: they only take part in the collective
            self.stream = self.engs[self.mine[0]].torch_stream() if self.mine else torch.cuda.current_stream(torch.device("cuda", device))
        tdev = torch.device("cuda", device) if self.on_cuda else torch.device("cpu")
        self.send = torch.zeros(self.width, dtype=torch.float64, device=tdev)
        self.recv = torch.zeros(world * self.width, dtype=torch.float64, device=tdev)
        self.arena = {s: self.engs[s].arena_tensor() for s in self.mine}             # complex128 views of the arenas
        self.slots = {s: self.engs[s].slots_tensor() for s in self.mine}
        # index tables: next iteration's message inputs of every local program <- gathered out blocks
        key = "next" if self.damping else "out"
        self.scatter = {}
        for s in self.mine:
            dst, src = [], []
            for name, off, shape in self.comps[s].in_layout:
                if not name.startswith("m"):
                    continue
                k = int("".join(ch for ch in name if ch.isdigit()))
                t = name[1:len(name) - len(str(k))]                  # message that sits on side t ...
                producer = SIDE_OPPOSITE[t]                           # ... was computed by the chain towards the opposite side
                lay = {nm: (q, sh) for nm, q, sh in self.comps[producer].out_layout}
                q, sh = lay[f"{key}{k}"]
                n = int(np.prod(shape))
                assert n == int(np.prod(sh)), (name, shape, sh)
                dst.append(np.arange(off, off + n, dtype=np.int64))
                src.append(self.pos[producer] // 2 + q + np.arange(n, dtype=np.int64))
                assert self.pos[producer] % 2 == 0
            self.scatter[s] = (torch.from_numpy(np.concatenate(dst)).to(tdev), torch.from_numpy(np.concatenate(src)).to(tdev))
        for s in BLOCK_SIDES_CCW:
            assert self.pos[s] % 2 == 0 and self.words[s] % 2 == 0, "complex view of the gathered buffer needs even offsets"
        self.events = {}
        if self.on_cuda:
            self.events = {s: torch.cuda.Event() for s in self.mine}
            self.done = torch.cuda.Event()

    def _pack_and_gather(self):
        torch = self.torch
        import torch.distributed as dist
        p = 0
        for s in self.mine:
            comp = self.comps[s]
            ob = self.arena[s][comp.out_block.off:comp.out_block.off + comp.out_elems]
            self.send[p:p + 2 * comp.out_elems].copy_(torch.view_as_real(ob).reshape(-1))
            self.send[p + 2 * comp.out_elems:p + self.words[s]].copy_(self.slots[s][:self.n_slots])
            p += self.words[s]
        dist.all_gather_into_tensor(self.recv, self.send, group=self.group)      # THE collective of a BP iteration
        recv_c = torch.view_as_complex(self.recv.reshape(-1, 2))
        for s in self.mine:
            dst, src = self.scatter[s]
            self.arena[s].index_copy_(0, dst, recv_c.index_select(0, src))

    def step(self):
        """one BP iteration; returns (error, trunc_error, status_ok) -- the same numbers on every rank."""
        torch = self.torch
        for s in self.mine:                                            # graph launches on the sides' own streams
            self.comps[s].run_resident(self.engs[s], (bp.E_SVD_NOCONV,))
        if self.on_cuda:
            main = self.stream
            for s in self.mine:
                ev = self.events[s]
                ev.record(self.engs[s].torch_stream())
                main.wait_event(ev)
            with torch.cuda.stream(main):
                self._pack_and_gather()
                self.done.record(main)
            for s in self.mine:                                        # the next launch on any local stream sees the new inputs
                self.engs[s].torch_stream().wait_event(self.done)
            sl = self._slot_rows().cpu().numpy()                        # tiny D2H: the BP loop's convergence test
        else:
            for s in self.mine:
                self.engs[s].sync()
            self._pack_and_gather()
            sl = self._slot_rows().numpy()
        dists, trunc = [], 0.0
        for k, s in enumerate(BLOCK_SIDES_CCW):
            row = sl[k]
            ip = complex(row[bp.SLOT_IP_RE], row[bp.SLOT_IP_IM])
            dists.append(max(0.0, 1.0 - abs(ip)))
            trunc += float(row[bp.SLOT_TRUNC])
        ok = bool(np.all(sl[:, -1] == 0) and np.all(sl[:, bp.SLOT_NONFINITE] == 0))
        if self.config.msg_diff_squared:
            err = sum(dists) / len(dists)
        else:
            err = float(np.sqrt(sum(dists)) / len(dists))
        return float(err), trunc, ok

    def _slot_rows(self):
        torch = self.torch
        idx = []
        for s in BLOCK_SIDES_CCW:
            base = self.pos[s] + 2 * self.comps[s].out_elems
            idx.append(torch.arange(base, base + self.n_slots))
        ii = torch.stack(idx).to(self.recv.device)
        if self.on_cuda:
            with torch.cuda.stream(self.stream):
                out = self.recv[ii]
            self.stream.synchronize()
            return out
        return self.recv[ii]

    def messages(self):
        """(out_messages, next_messages) of the last iteration as host objects (any rank: everything was gathered)."""
        from .containers import Message, MPSOrientation
        from .mps import MPS
        flat = self.recv.cpu().numpy()
        out_msgs, next_msgs = {}, {}
        for s in BLOCK_SIDES_CCW:
            comp = self.comps[s]
            blk = flat[self.pos[s]:self.pos[s] + 2 * comp.out_elems].view(np.complex128)
            lay = {nm: (q, sh) for nm, q, sh in comp.out_layout}
            n_out = sum(1 for nm in lay if nm.startswith("out"))
            opp = SIDE_OPPOSITE[s]

            def sites(key):
                return [blk[lay[f"{key}{k}"][0]:lay[f"{key}{k}"][0] + int(np.prod(lay[f"{key}{k}"][1]))].reshape(lay[f"{key}{k}"][1]).copy()
                        for k in range(n_out)]
            orient = MPSOrientation.standard(s)
            out_msgs[opp] = Message(MPS.from_sites(sites("out"), Corder=[None] + ["R"] * (n_out - 1)), orient)
            if self.damping:
                next_msgs[opp] = Message(MPS.from_sites(sites("next"), Corder=[None] + ["R"] * (n_out - 1)), orient)
        return out_msgs, (next_msgs if self.damping else out_msgs)


def bp_step_sharded(N: int, cells: list, messages_list: list, config, rank: int, world: int, device: int = 0, group=None,
                    torch_device=None):
    """one BP iteration of ONE cell with the six sides sharded over ``world`` ranks (stateless convenience wrapper around
    ``ShardedSides``: uploads the messages, runs one step, returns host objects).  Every rank returns the same
    [(out_messages, next_messages, error, trunc_error)], gathered bytes."""
    assert len(cells) == 1, "side sharding is for one unit cell; ensembles shard by cells"
    sh = ShardedSides(N, cells[0], messages_list[0], config, rank, world, device, group)
    err, trunc, ok = sh.step()
    if not ok:
        raise bp.BubbleConError("sharded BP step: a truncation did not converge or produced non-finite values on some rank")
    out_msgs, next_msgs = sh.messages()
    return [(out_msgs, next_msgs, err, trunc)], sh.gather_bytes


def gather_scalars(values, world: int, group=None, torch_device=None):
    """all ranks' scalar results (energies, errors) on every rank."""
    import torch
    import torch.distributed as dist
    dev = torch_device if torch_device is not None else "cpu"
    send = torch.tensor(list(values), dtype=torch.float64, device=dev)
    recv = [torch.empty_like(send) for _ in range(world)]
    dist.all_gather(recv, send, group=group)
    return [r.cpu().numpy() for r in recv]
