"""Slab decomposition of the solve across the GPUs of one box (one process per GPU, torch.distributed).

The grid rows (x2 index, the sweep direction of algo2_4, /root/reference/code.py:356-385) are cut into
contiguous slabs, rank r owns rows R[r] .. R[r+1]-1 (0-based).  Per rank:
  * Krylov vectors hold the rank's rows only; dot products are all-reduced              (NCCL / gloo)
  * the stencil matvec needs one halo row from each neighbour                            (send/recv)
  * strip T_m (b+1 <= m <= n) lives with its input row m-1, so rank r factors and applies the strips
    m = R[r]+1 .. R[r+1]; the front block H_F lives on rank 0 (which must own rows 0..b)
  * the sweeps are a chain over the strips, hence over the ranks: the forward sweep hands the updated first
    row of the next slab downstream, the backward sweep hands the final first row upstream.  Only one rank
    sweeps at a time - the decomposition buys memory capacity (the strip factors dominate), not sweep speed.

`backend` is the per-rank compute object: HelmholtzSolver on a GPU, or any object with the same staged
methods (the CPU tests drive the message schedule with a numpy stand-in over gloo).
"""
import os

import numpy as np
import torch
import torch.distributed as dist

from .gmres import CommStats

os.environ.setdefault("TORCH_NCCL_SHOW_EAGER_INIT_P2P_SERIALIZATION_WARNING", "false")


def slab_bounds(n, b, world, front_equiv=0):
    """R[0..world]: rank r owns rows R[r]..R[r+1]-1.  Rank 0 must own rows 0..b (front block + row b).
    front_equiv > 0 balances the pipelined sweeps: the front solves of rank 0 cost as much as that many strips, so
    rank 0 gets that many strips less than its share (strip m belongs to the owner of row m-1)."""
    if front_equiv <= 0 or world == 1:
        R = [(n * r) // world for r in range(world + 1)]
    else:
        strips = n - b                                        # m = b+1..n, inputs in rows b..n-1
        share = (strips + front_equiv) / world
        first = max(1, min(strips - (world - 1), int(round(share - front_equiv))))   # strips of rank 0
        rest = strips - first
        R = [0] + [b + first + (rest * r) // (world - 1) for r in range(world)]
        R[-1] = n
    if world > 1 and R[1] < b + 1:
        raise ValueError(f"slab of rank 0 ({R[1]} rows) must contain the front block and one more row ({b + 1} rows)")
    return R


class SlabSolver:
    """Distributed operator/preconditioner on slab-distributed vectors (local shape (rows, n), flattened)."""

    def __init__(self, backend, n, b, rank, world, group=None, device="cpu", front_equiv=0):
        self.s, self.n, self.b, self.rank, self.world, self.group = backend, n, b, rank, world, group
        self.R = slab_bounds(n, b, world, front_equiv)
        self.j0, self.j1 = self.R[rank], self.R[rank + 1]
        self.rows = self.j1 - self.j0
        self.device = device
        # strips of this rank: m-1 in [j0, j1)  ->  m in [j0+1, j1], clipped to b+1..n
        self.m_lo, self.m_hi = max(b + 1, self.j0 + 1), min(n, self.j1)
        # local work buffer with one ghost row below (row j0-1) and above (row j1)
        self.buf = torch.zeros((self.rows + 2) * n, dtype=torch.complex128, device=device)
        self.bufs, self.tfs = [self.buf], []                 # work buffers / parked T_F u_F of a batch of right-hand sides
        self.south = torch.zeros(n, dtype=torch.complex128, device=device)
        self.north = torch.zeros(n, dtype=torch.complex128, device=device)
        self.halos = []                                      # halo rows of a batch of systems (matvec_batch)
        self.mail, self.seq = None, 0                        # PeerMailbox of this solver (GroupPipeline), applications so far

    # -- communication helpers ------------------------------------------------------------------------
    def _send(self, t, dst):
        CommStats.calls += 1
        dist.send(t.contiguous(), dst, group=self.group)

    def _recv(self, t, src):
        CommStats.calls += 1
        dist.recv(t, src, group=self.group)

    def _isend(self, t, dst):
        CommStats.calls += 1
        return dist.isend(t, dst, group=self.group)

    def _exchange(self, ops):
        """one batched non-blocking exchange (a single NCCL group call)"""
        if not ops:
            return
        CommStats.calls += 1
        for q in dist.batch_isend_irecv(ops):
            q.wait()

    def _post(self, ops):
        """batched non-blocking sends that the caller waits for later; returns their work handles"""
        CommStats.calls += 1
        return dist.batch_isend_irecv(ops)

    def _row(self, j, buf=None):
        """view of global row j inside the ghosted buffer (j0-1 <= j <= j1)."""
        o = (j - (self.j0 - 1)) * self.n
        return (self.buf if buf is None else buf)[o:o + self.n]

    # -- operator -------------------------------------------------------------------------------------
    def matvec(self, x, out):
        """out = A x on the slab; exchanges the boundary rows with the neighbours first."""
        n, r, w = self.n, self.rank, self.world
        first, last = x[:n], x[(self.rows - 1) * n:]
        if w > 1:
            ops = []
            if r > 0:
                ops += [dist.P2POp(dist.isend, first.contiguous(), r - 1, self.group), dist.P2POp(dist.irecv, self.south, r - 1, self.group)]
            if r < w - 1:
                ops += [dist.P2POp(dist.isend, last.contiguous(), r + 1, self.group), dist.P2POp(dist.irecv, self.north, r + 1, self.group)]
            self._exchange(ops)
        self.s.matvec_rows(self.j0, self.j1, x, self.south if r > 0 else None, self.north if r < w - 1 else None, out)
        return out

    def matvec_batch(self, pairs):
        """out_i = A x_i for several systems: the halo rows of all of them travel in one exchange"""
        n, r, w = self.n, self.rank, self.world
        R = len(pairs)
        while len(self.halos) < R:
            self.halos.append((torch.zeros_like(self.south), torch.zeros_like(self.north)))
        if w > 1:
            ops = []
            for i, (x, _) in enumerate(pairs):
                so, no = self.halos[i]
                if r > 0:
                    ops += [dist.P2POp(dist.isend, x[:n], r - 1, self.group), dist.P2POp(dist.irecv, so, r - 1, self.group)]
                if r < w - 1:
                    ops += [dist.P2POp(dist.isend, x[(self.rows - 1) * n:], r + 1, self.group), dist.P2POp(dist.irecv, no, r + 1, self.group)]
            self._exchange(ops)
        for i, (x, out) in enumerate(pairs):
            so, no = self.halos[i]
            self.s.matvec_rows(self.j0, self.j1, x, so if r > 0 else None, no if r < w - 1 else None, out)

    # -- preconditioner -------------------------------------------------------------------------------
    def precond_apply(self, x, out, diag="reference"):
        """out = M x (algo2_4) on slab-distributed vectors."""
        n, b, r, w = self.n, self.b, self.rank, self.world
        own = self.buf[n:(self.rows + 1) * n]
        own.copy_(x)
        buf, row0 = self.buf, self.j0 - 1                    # the buffer starts at global row j0-1
        # ghost row above = first row of the next slab (initial values: the forward sweep updates it)
        if r > 0:
            self._send(own[:n], r - 1)
        if r < w - 1:
            self._recv(self._row(self.j1), r + 1)
        # forward chain
        if r == 0:
            self.s.front_begin_buf(buf, row0)
        else:
            self._recv(self._row(self.j0), r - 1)            # first own row, updated by the previous rank
        m_to = min(self.m_hi, n - 1)
        if self.m_lo <= m_to:
            self.s.sweep_forward_buf(buf, row0, self.m_lo, m_to)
        if r < w - 1:
            self._send(self._row(self.j1), r + 1)
        # backward chain
        if r < w - 1:
            self._recv(self._row(self.j1), r + 1)            # final first row of the next slab
        if self.m_lo <= self.m_hi:
            self.s.sweep_backward_buf(buf, row0, self.m_hi, self.m_lo, diag)
        if r > 0:
            self._send(self._row(self.j0), r - 1)
        else:
            self.s.front_end_buf(buf, row0)
        out.copy_(own)
        return out


    def batch_group(self, R):
        """right-hand sides one sweep launch carries when R are in flight (the multi-vector kernels of the backend)"""
        return self.s.batch_group(R) if hasattr(self.s, "batch_group") else 1

    def precond_apply_batch(self, pairs, diag="reference"):
        """out_i = M x_i for every (x_i, out_i) of `pairs`.  The right-hand sides travel through the slabs in groups: a group
        is swept by ONE launch of the multi-vector kernel per slab (the strip generators are streamed once for the whole
        group), and the groups follow each other through the slabs: while rank r sweeps its strips for group j, rank
        r+1 sweeps them for group j-1.  Per sweep direction G groups take (world - 1 + G) slab sweeps instead of G * world;
        the rows handed over are posted as non-blocking sends so that a rank goes on with the next group at once."""
        n, b, r, w = self.n, self.b, self.rank, self.world
        R = len(pairs)
        if self.mail is not None and w > 1:
            return self._precond_apply_batch_mailbox(pairs, diag)
        while len(self.bufs) < R:
            self.bufs.append(torch.zeros_like(self.buf))
        if r == 0 and hasattr(self.s, "front_tf_new"):
            while len(self.tfs) < R:
                self.tfs.append(self.s.front_tf_new())
        row0 = self.j0 - 1
        owns = [self.bufs[i][n:(self.rows + 1) * n] for i in range(R)]
        for i, (x, _) in enumerate(pairs):
            owns[i].copy_(x)
        # ghost rows above (initial values of the first row of the next slab), all right-hand sides in one exchange
        if w > 1:
            ops = []
            for i in range(R):
                if r > 0:
                    ops.append(dist.P2POp(dist.isend, owns[i][:n], r - 1, self.group))
                if r < w - 1:
                    ops.append(dist.P2POp(dist.irecv, self._row(self.j1, self.bufs[i]), r + 1, self.group))
            self._exchange(ops)
        groups, i = [], 0
        while i < R:
            g = self.batch_group(R - i)
            groups.append(list(range(i, i + g)))
            i += g
        multi = hasattr(self.s, "sweep_forward_multi_buf")
        sends = []
        m_to = min(self.m_hi, n - 1)
        for grp in groups:                                   # forward chain
            bufs = [self.bufs[i] for i in grp]
            for i in grp:
                if r == 0:
                    self.s.front_begin_buf(self.bufs[i], row0)
                    if R > 1:
                        self.s.front_tf_save(self.tfs[i])
            if r > 0:
                self._exchange([dist.P2POp(dist.irecv, self._row(self.j0, bf), r - 1, self.group) for bf in bufs])
            if self.m_lo <= m_to:
                if multi and len(grp) > 1:
                    self.s.sweep_forward_multi_buf(bufs, row0, self.m_lo, m_to)
                else:
                    for bf in bufs:
                        self.s.sweep_forward_buf(bf, row0, self.m_lo, m_to)
            if r < w - 1:
                sends += self._post([dist.P2POp(dist.isend, self._row(self.j1, bf), r + 1, self.group) for bf in bufs])
        for q in sends:                                      # the rows come back in the backward chain
            q.wait()
        sends = []
        for grp in groups:                                   # backward chain
            bufs = [self.bufs[i] for i in grp]
            if r < w - 1:
                self._exchange([dist.P2POp(dist.irecv, self._row(self.j1, bf), r + 1, self.group) for bf in bufs])
            if self.m_lo <= self.m_hi:
                if multi and len(grp) > 1:
                    self.s.sweep_backward_multi_buf(bufs, row0, self.m_hi, self.m_lo, diag)
                else:
                    for bf in bufs:
                        self.s.sweep_backward_buf(bf, row0, self.m_hi, self.m_lo, diag)
            if r > 0:
                sends += self._post([dist.P2POp(dist.isend, self._row(self.j0, bf), r - 1, self.group) for bf in bufs])
            else:
                for i in grp:
                    if R > 1:
                        self.s.front_tf_load(self.tfs[i])
                    self.s.front_end_buf(self.bufs[i], row0)
        for q in sends:
            q.wait()
        for i, (_, out) in enumerate(pairs):
            out.copy_(owns[i])


    def _precond_apply_batch_mailbox(self, pairs, diag):
        """precond_apply_batch with the rows handed over through peer mailboxes (PeerMailbox): up to 8 right-hand sides that
        travel together.  Between the sweeps of this rank and those of its neighbours no communication kernel waits on the
        device: the stream waits for sequence numbers (application count `seq`) that the neighbour releases after its rows
        have been stored into this rank's staging area.  Ranks > 0 leave the application only when rank 0 has finished
        it, so that every collective that follows (halo exchange, dot products) finds all ranks in their vector phase."""
        n, b, r, w, mail = self.n, self.b, self.rank, self.world, self.mail
        R = len(pairs)
        assert R <= mail.R, "a mailbox carries the rows of one group of right-hand sides"
        self.seq += 1
        seq = self.seq
        while len(self.bufs) < R:
            self.bufs.append(torch.zeros_like(self.buf))
        if r == 0:
            while len(self.tfs) < R:
                self.tfs.append(self.s.front_tf_new())
        row0 = self.j0 - 1
        bufs = self.bufs[:R]
        owns = [bf[n:(self.rows + 1) * n] for bf in bufs]
        for i, (x, _) in enumerate(pairs):
            owns[i].copy_(x)
        ops = []                                             # ghost rows above: initial values of the first row of the next slab
        for i in range(R):
            if r > 0:
                ops.append(dist.P2POp(dist.isend, owns[i][:n], r - 1, self.group))
            if r < w - 1:
                ops.append(dist.P2POp(dist.irecv, self._row(self.j1, bufs[i]), r + 1, self.group))
        self._exchange(ops)
        groups, i = [], 0
        while i < R:
            g = self.batch_group(R - i)
            groups.append(list(range(i, i + g)))
            i += g
        m_to = min(self.m_hi, n - 1)
        # forward chain
        if r == 0:
            for i in range(R):
                self.s.front_begin_buf(bufs[i], row0)
                if R > 1:
                    self.s.front_tf_save(self.tfs[i])
        else:
            mail.wait(mail.FWD, seq)
            mail.collect(mail.FWD, [self._row(self.j0, bf) for bf in bufs])
        if self.m_lo <= m_to:
            for grp in groups:
                if len(grp) > 1:
                    self.s.sweep_forward_multi_buf([bufs[i] for i in grp], row0, self.m_lo, m_to)
                else:
                    self.s.sweep_forward_buf(bufs[grp[0]], row0, self.m_lo, m_to)
        if r < w - 1:
            mail.handover(r + 1, mail.FWD, [self._row(self.j1, bf) for bf in bufs], seq)
            # backward chain
            mail.wait(mail.BWD, seq)
            mail.collect(mail.BWD, [self._row(self.j1, bf) for bf in bufs])
        if self.m_lo <= self.m_hi:
            for grp in groups:
                if len(grp) > 1:
                    self.s.sweep_backward_multi_buf([bufs[i] for i in grp], row0, self.m_hi, self.m_lo, diag)
                else:
                    self.s.sweep_backward_buf(bufs[grp[0]], row0, self.m_hi, self.m_lo, diag)
        if r > 0:
            mail.handover(r - 1, mail.BWD, [self._row(self.j0, bf) for bf in bufs], seq)
            mail.wait(mail.DONE, seq)
        else:
            for i in range(R):
                if R > 1:
                    self.s.front_tf_load(self.tfs[i])
                self.s.front_end_buf(bufs[i], row0)
            mail.signal_done(seq)
        for i, (_, out) in enumerate(pairs):
            out.copy_(owns[i])


class PeerMailbox:
    """Staging rows and sequence numbers of one group of right-hand sides on this rank, mapped by the neighbouring ranks
    through CUDA IPC (csrc/hp_peer.cu): [256 bytes of flags | forward staging [R][n] | backward staging [R][n]].
    Built collectively: create() on every rank, exchange of the handles, connect()."""
    FWD, BWD, DONE = 0, 1, 2

    def __init__(self, n, R, device):
        import ctypes as C
        from . import _lib
        self.lib = _lib.require_device()
        self.C, self.check = C, _lib.check
        self.n, self.R, self.device = n, R, device
        self.bytes = 256 + 2 * R * n * 16
        ptr, handle = C.c_void_p(), (C.c_ubyte * 64)()
        with torch.cuda.device(device):
            self.check(self.lib.hp_mailbox_create(self.bytes, C.byref(ptr), handle), "hp_mailbox_create")
        self.ptr, self.handle = ptr.value, bytes(handle)
        self.peers = {}                                      # rank -> device address of that rank's mailbox in this process

    def connect(self, handles, rank, world):
        """handles[r]: the 64-byte handle of rank r's mailbox.  Neighbours map each other; rank 0 maps everybody (DONE)."""
        C = self.C
        self.rank, self.world = rank, world
        need = {rank - 1, rank + 1} if rank > 0 else set(range(1, world))
        with torch.cuda.device(self.device):
            for p in sorted(q for q in need if 0 <= q < world and q != rank):
                ptr = C.c_void_p()
                h = (C.c_ubyte * 64).from_buffer_copy(handles[p])
                self.check(self.lib.hp_mailbox_open(h, C.byref(ptr)), "hp_mailbox_open")
                self.peers[p] = ptr.value

    def _stream(self):
        return torch.cuda.current_stream().cuda_stream

    def _staging(self, base, which):
        return base + 256 + which * self.R * self.n * 16

    def wait(self, which, seq):
        self.check(self.lib.hp_stream_wait_geq(self.ptr + 4 * which, seq, self._stream()), "hp_stream_wait_geq")

    def collect(self, which, rows):
        arr = (self.C.c_void_p * len(rows))(*[t.data_ptr() for t in rows])
        self.check(self.lib.hp_collect_rows(len(rows), self._staging(self.ptr, which), arr, self.n, self._stream()), "hp_collect_rows")

    def handover(self, peer, which, rows, seq):
        base = self.peers[peer]
        arr = (self.C.c_void_p * len(rows))(*[t.data_ptr() for t in rows])
        self.check(self.lib.hp_handover_rows(len(rows), arr, self._staging(base, which), self.n, base + 4 * which, seq, self._stream()),
                   "hp_handover_rows")

    def signal_done(self, seq):
        ranks = [p for p in sorted(self.peers) if p > 0]
        for i in range(0, len(ranks), 8):
            chunk = ranks[i:i + 8]
            arr = (self.C.c_void_p * len(chunk))(*[self.peers[p] + 4 * self.DONE for p in chunk])
            self.check(self.lib.hp_signal_flags(len(chunk), arr, seq, self._stream()), "hp_signal_flags")

    def close(self):
        with torch.cuda.device(self.device):
            for p in self.peers.values():
                self.lib.hp_mailbox_close(p)
            self.peers = {}
            if self.ptr:
                self.lib.hp_mailbox_free(self.ptr)
                self.ptr = None


def distributed_gmres_setup(n, b, omega, const, c_mat, rank, world, group, device, P=0, K=0, front_equiv=0):
    """HelmholtzSolver of this rank with its strips factored, wrapped in a SlabSolver."""
    from .solver import HelmholtzSolver
    s = HelmholtzSolver(n, b, omega, const, c_mat, device=device)
    R = slab_bounds(n, b, world, front_equiv)
    m_lo, m_hi = max(b + 1, R[rank] + 1), min(n, R[rank + 1])
    s.setup_preconditioner(P, K, m_lo, m_hi)
    return SlabSolver(s, n, b, rank, world, group, device=device, front_equiv=front_equiv)


class GroupPipeline:
    """Groups of right-hand sides that run through the slabs independently of each other.

    precond_apply_batch/gmres_batch advance all right-hand sides in lock step: every sweep direction of every Krylov
    iteration fills and drains the chain of slabs, G groups take (world - 1 + G) slab sweeps per direction and a rank is
    busy G / (world - 1 + G) of the time.  Here every group of right-hand sides (one launch of the multi-vector sweep
    kernel per slab and direction) is an independent restarted GMRES with its own
      * host thread (runs gmres_batch on the systems of the group and blocks on its own results only),
      * CUDA stream (the device takes the next ready kernel of any group: a greedy list schedule of the slab sweeps),
      * solver context (HelmholtzSolver.clone_context: private exchange ring / abort flags / parked front solutions),
      * process group (its own communicator, so that no order of calls has to be kept between the groups).
    A group starts its next iteration as soon as its own backward sweep has reached rank 0, while the other groups are
    anywhere in their sweeps: in the steady state a rank always has a slab sweep or the vector work of some group to
    run as soon as there are about as many groups as ranks.  The arithmetic of a system is that of gmres_batch on its
    group alone: results do not depend on how the groups interleave.

    Device-side progress.  The cluster sweep kernels need every cluster slot of the GPU (33 clusters of 4 whole SMs at
    4096^2), so a communication kernel that spins on an SM while it waits for a sweep on ANOTHER GPU can keep a sweep of
    another group partially resident on THIS GPU, and two GPUs can wait for each other that way (measured: the schedule
    with NCCL receives for the rows hangs at N = 2).  Therefore (i) the rows travel through PeerMailbox: stores into the
    neighbour's memory and stream-level waits for sequence numbers, no kernel waits for a sweep; (ii) ranks > 0 leave an
    application of the preconditioner only when rank 0 has finished it, so the NCCL kernels that remain (ghost rows at the
    start of an application, halo rows of the matvec, dot products; one CTA each, pg_options below) only ever wait for
    vector kernels of the same group on the other ranks, which always find a free SM.
    """

    def __init__(self, S, n_groups, device=None, backend="nccl", streams=True, rhs_per_group=8, mailboxes=True, solver_cls=None):
        self.S, self.G = S, int(n_groups)
        self.device = S.device if device is None else device
        self.cuda = torch.device(self.device).type == "cuda"
        self.members = []
        self.mails = []
        self.primed = False
        if self.cuda and S.world > 1 and mailboxes:         # row hand-over through peer memory (see PeerMailbox)
            self.mails = [PeerMailbox(S.n, rhs_per_group, self.device) for _ in range(self.G)]
            handles = [None] * S.world
            dist.all_gather_object(handles, [m.handle for m in self.mails])
            for g, m in enumerate(self.mails):
                m.connect([handles[r][g] for r in range(S.world)], S.rank, S.world)
        for g in range(self.G):
            pg = None
            if S.world > 1:
                opts = None
                if backend == "nccl":
                    opts = dist.ProcessGroupNCCL.Options()
                    opts.config.min_ctas = 1
                    opts.config.max_ctas = 1
                    opts.config.cga_cluster_size = 1
                pg = dist.new_group(backend=backend, pg_options=opts) if opts is not None else dist.new_group(backend=backend)
            ctx = S.s.clone_context() if hasattr(S.s, "clone_context") else S.s
            Sg = (solver_cls or SlabSolver)(ctx, S.n, S.b, S.rank, S.world, pg, device=self.device)
            Sg.R, Sg.j0, Sg.j1, Sg.rows, Sg.m_lo, Sg.m_hi = S.R, S.j0, S.j1, S.rows, S.m_lo, S.m_hi
            Sg.mail = self.mails[g] if self.mails else None
            stream = torch.cuda.Stream(device=self.device) if (self.cuda and streams) else None
            self.members.append((Sg, pg, stream))

    def close(self):
        if self.mails:
            torch.cuda.synchronize()
            dist.barrier()                                   # nobody writes into a mailbox any more
            for m in self.mails:
                m.close()
            self.mails = []
        for Sg, pg, _ in self.members:
            if Sg.s is not self.S.s and hasattr(Sg.s, "close"):
                Sg.s.close()
            if pg is not None:
                dist.destroy_process_group(pg)
        self.members = []

    def sweep_status(self):
        return max([int(Sg.s.sweep_status()) for Sg, _, _ in self.members if hasattr(Sg.s, "sweep_status")] + [0])

    def gmres(self, rhs_groups, make_vec, *, diag="reference", host_out=None, **kw):
        """rhs_groups[g]: list of local right-hand side slabs of group g; make_vec(nloc, process_group) -> the vector
        kernels of a group (gmres.DeviceVectors on a GPU).  Returns [[(x, info, hist), ...] per group].
        Right-hand sides given as (pinned) host tensors are copied to the device on the group's own stream, and with
        host_out[g] = [pinned host tensor per system] the solutions go back the same way: the transfers of one group
        overlap the sweeps of the others."""
        import contextlib
        import sys
        import threading
        from .gmres import gmres_batch
        assert len(rhs_groups) == self.G
        results, errors = [None] * self.G, [None] * self.G
        start = torch.cuda.Event() if self.cuda else None

        def work(g, out, kwg):
            Sg, pg, stream = self.members[g]
            try:
                with (torch.cuda.device(self.device) if self.cuda else contextlib.nullcontext()):
                    with (torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()):
                        if stream is not None:
                            stream.wait_event(start)
                        vec = make_vec(rhs_groups[g][0].numel(), pg)
                        rhs = [t.to(self.device, non_blocking=True) if (self.cuda and not t.is_cuda) else t for t in rhs_groups[g]]
                        out[g] = gmres_batch(lambda x, o: Sg.matvec(x, o), lambda reqs: Sg.precond_apply_batch(reqs, diag=diag),
                                             rhs, vec=vec, matvec_batch=lambda reqs: Sg.matvec_batch(reqs), **kwg)
                        if host_out is not None and out is results:
                            for uh, (x, _, _) in zip(host_out[g], out[g]):
                                uh.copy_(x, non_blocking=True)
                        if stream is not None:
                            stream.synchronize()
            except BaseException as e:                       # noqa: B902 - re-raised by the caller's thread
                import traceback
                traceback.print_exc()                        # at once: the other groups/ranks may now wait for this one for ever
                errors[g] = e

        if not self.primed:
            # Every group runs two iterations ALONE first, one group after the other on all ranks.  With lazy module loading
            # (the CUDA 12 default) the first launch of a kernel may synchronise the whole context; once streams of this
            # process wait for other GPUs that is a deadlock (measured: rank 1 blocked inside its first launch of the collect
            # kernel behind the pending wait of another group, rank 0 likewise).  The pass also connects the communicator of
            # every group and lets the contexts and the caching allocator of every stream make their allocations.
            if start is not None:
                start.record()
            prime = dict(kw, rtol=0.0, atol=0.0, maxiter=2, callback=None)
            for g in range(self.G):
                work(g, [None] * self.G, prime)
                if errors[g] is not None:
                    raise errors[g]
            self.primed = True
        if start is not None:
            start.record()                                   # the groups start after what the caller has enqueued

        old = sys.getswitchinterval()
        sys.setswitchinterval(1e-4)                          # a thread whose result has arrived should not wait 5 ms for the GIL
        try:
            threads = [threading.Thread(target=work, args=(g, results, kw), name=f"hp-group-{g}") for g in range(self.G)]
            for t in threads:
                t.start()
            for t in threads:
                t.join()
        finally:
            sys.setswitchinterval(old)
        for e in errors:
            if e is not None:
                raise e
        if self.cuda:
            for _, _, stream in self.members:
                if stream is not None:
                    torch.cuda.current_stream().wait_stream(stream)
        return results
