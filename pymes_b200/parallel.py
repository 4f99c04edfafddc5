"""Sharding of the coupled-cluster iteration over the GPUs of one box.

One process per GPU (torchrun); ``torch.distributed`` (NCCL over NVLink on the box, gloo in
the CPU tests) is the plumbing.  The composite virtual-pair index (ab) of every [a,b,i,j]
quantity and of V_abcd[(ab),(cd)] is split into contiguous row blocks over its leading index a
(SURVEY 8e): rank r owns a in [r*mr, min((r+1)*mr, nv)), mr = ceil(nv / n_ranks).

Per rank (LOCAL row blocks)      V_abcd[A,:,:,:], V_abci[A], V_abic[A], V_aibc[A], V_iabc[:,A]
                                 -- the v^4 / o.v^3 blocks, i.e. everything that is big
replicated                       T1, T2, Fock and every o^2v^2 / o^3v / o^4 block

Exchange steps of one CCSD iteration (all over NVLink, none on the O(o^2v^4) data path):
  * all-gather of the new T2 row blocks                      (o^2v^2 * 8 B in total)
  * all-gather of Ex for the explicit Ex + Ex^{baji}          (o^2v^2 * 8 B)
  * all-gather of the ring intermediate Xai, of the two T1-dressed o^2v^2 blocks and of the
    o^3v-sized W1 of the tau ladder
  * one all-reduce of the scalar pack (E_dir, E_ex, |T2|^2, |dT2|^2) and one of the DIIS row.
The ladder / ring contractions themselves never communicate.
"""
import math

import numpy as np
import torch
import torch.distributed as dist

from . import backend as bk
from .solver import ccd, ccsd, mp2
from .solver.ccsd import FOCK_SHARED, FOCK_TERMS, SHARED_PRODUCTS, V_TERMS, SINGLES_TERMS

# integral blocks held as local row blocks: key -> dimension that carries the sharded index
# (the o^2v^2 blocks V_aibj / V_aijb are read by two rows of the dressed V_abij only, always with a
#  as the row index: held as local rows as well -- 5 GB each at o = 50, v = 500)
SHARD_DIMS = {"abcd": 0, "abci": 0, "abic": 0, "aibc": 0, "iabc": 1, "aibj": 0, "aijb": 0}


class Comm:
    """Thin wrapper over a torch.distributed process group."""

    def __init__(self, group=None):
        self.group = group
        self.rank = dist.get_rank(group)
        self.size = dist.get_world_size(group)

    def all_gather_rows(self, local, n_rows, max_rows):
        """local [na, ...] (this rank's rows) -> [n_rows, ...] with every rank's rows in order.
        All ranks but the last own exactly ``max_rows`` rows, so the gathered buffer
        [size*max_rows, ...] holds the full tensor as a contiguous prefix (no reassembly copy)."""
        rest = tuple(local.shape[1:])
        send = local.contiguous()
        if send.shape[0] != max_rows:
            pad = torch.zeros((max_rows,) + rest, dtype=local.dtype, device=local.device)
            pad[: send.shape[0]] = send
            send = pad
        buf = torch.empty((self.size * max_rows,) + rest, dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(buf, send, group=self.group)
        return buf[:n_rows]

    def all_gather_rows_async(self, local, n_rows, max_rows):
        """Same as :meth:`all_gather_rows`, started now and completed by ``.wait_result()``: the
        collective runs on the communicator's own stream while the caller keeps launching
        independent kernels on the compute stream."""
        rest = tuple(local.shape[1:])
        send = local.contiguous()
        if send.shape[0] != max_rows:
            pad = torch.zeros((max_rows,) + rest, dtype=local.dtype, device=local.device)
            pad[: send.shape[0]] = send
            send = pad
        buf = torch.empty((self.size * max_rows,) + rest, dtype=local.dtype, device=local.device)
        work = dist.all_gather_into_tensor(buf, send, group=self.group, async_op=True)
        return Pending(work, buf[:n_rows], keep=(send,))

    def exchange_blocks(self, send):
        """send [size, ...]: block q goes to rank q; returns recv [size, ...] with block q coming
        from rank q (all-to-all, equal blocks)."""
        send = send.contiguous()
        recv = torch.empty_like(send)
        dist.all_to_all_single(recv, send, group=self.group)
        return recv

    def all_reduce_sum(self, x):
        """numpy array or tensor, summed over ranks (returned in the same kind)."""
        if isinstance(x, np.ndarray):
            t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(bk.device())
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
            return t.cpu().numpy()
        dist.all_reduce(x, op=dist.ReduceOp.SUM, group=self.group)
        return x

    def barrier(self):
        dist.barrier(group=self.group)


class Pending:
    """Result of a collective that is still in flight."""

    def __init__(self, work, result, keep=(), view=None):
        self.work, self.result, self.keep, self.view = work, result, keep, view

    def wait_result(self):
        if self.work is not None:
            self.work.wait()          # the compute stream waits; the host does not
            self.work, self.keep = None, ()
        return self.view(self.result) if self.view is not None else self.result


def resolved(x):
    """A tensor, or the tensor a :class:`Pending` collective delivers."""
    return x.wait_result() if isinstance(x, Pending) else x


class Shard:
    """Row block [lo, lo+na) of an index of extent nv owned by this rank."""

    def __init__(self, comm, nv):
        self.comm, self.nv, self.size = comm, nv, comm.size
        self.max_rows = int(math.ceil(nv / comm.size))
        self.lo = min(comm.rank * self.max_rows, nv)
        self.na = min(self.lo + self.max_rows, nv) - self.lo
        if (comm.size - 1) * self.max_rows >= nv:
            raise ValueError("%d virtual orbitals cannot be split into %d non-empty row blocks"
                             % (nv, comm.size))

    def rows(self, t, dim=0):
        return bk.narrow(t, dim, self.lo, self.na)       # keeps the geometry tag of a stored V block

    def gather(self, local):
        return self.comm.all_gather_rows(local, self.nv, self.max_rows)

    def gather_async(self, local, view=None):
        p = self.comm.all_gather_rows_async(local, self.nv, self.max_rows)
        p.view = view
        return p

    def transposed_rows(self, Ex):
        """Ex [na, nv, o, o] (this rank's rows a of an [a,b,i,j] tensor) -> the rows a in A of its
        (ba)(ji) transpose, T[a,b,i,j] = Ex_full[b,a,j,i], as a VIEW [na, nv, o, o].  Rank q owns
        the rows b in A_q of Ex_full, so it sends its columns a in A_me: an all-to-all of
        o^2 v^2 / N elements per rank (the all-gather of Ex moves N times as much)."""
        mr, na, size = self.max_rows, self.na, self.size
        no = Ex.shape[2]
        send = torch.zeros((size, mr, mr, no, no), dtype=Ex.dtype, device=Ex.device)
        for q in range(size):
            lo = q * mr
            n = min(lo + mr, self.nv) - lo
            bk.axpby(1.0, Ex[:, lo:lo + n], 0.0, send[q, :na, :n])
        recv = self.comm.exchange_blocks(send)      # recv[q, b', a', j, i] = Ex_q[b', a_me + a', j, i]
        full = recv.reshape(size * mr, mr, no, no)  # [b (global, padded), a', j, i]
        return full.permute(1, 0, 3, 2)[:na, :self.nv]

    def all_reduce(self, x):
        """Sum of a small replicated-size tensor over the ranks (in place)."""
        return self.comm.all_reduce_sum(x)

    def gather_dim1(self, local_rows_first):
        """local [na, x, ...] holding block [x, A, ...] transposed -> full view [x, nv, ...]."""
        return self.gather(local_rows_first).transpose(0, 1)


def shard_blocks(dV_full, shard):
    """Slice a full integral dictionary into what one rank holds (tests / small systems)."""
    out = {}
    for k, v in dV_full.items():
        if v is None:
            out[k] = None
        elif k in SHARD_DIMS:
            out[k] = shard.rows(v, SHARD_DIMS[k])
        else:
            out[k] = v
    return out


def build_sharded_hamiltonian(m, no, comm, parts, virtual=()):
    """UEG integral blocks built directly as this rank's row blocks (no communication):
    the v^4 / o.v^3 blocks only for a in [lo, lo+na).  ``parts`` and ``virtual`` (keys kept as
    never-materialised operands, e.g. ``("abcd",)``) as in UEG.eval_2b_blocks."""
    from .integral.partition import KEYS
    nv = m.n_orb - no
    shard = Shard(comm, nv)
    ranges = {k: {SHARD_DIMS[k]: (no + shard.lo, shard.na)} for k in SHARD_DIMS}
    return m.eval_2b_blocks(no, list(KEYS), parts, ranges=ranges, virtual=virtual)


class ShardedCCSD(ccsd.CCSD):
    """CCSD / DCSD with the (ab) row blocks of the residual spread over the ranks of ``comm``.
    Same ``setup`` / ``sweep`` / ``solve`` interface as :class:`pymes_b200.solver.ccsd.CCSD`;
    the integral dictionary passed in holds LOCAL row blocks for the keys in ``SHARD_DIMS``."""

    def __init__(self, no, comm, **kw):
        super().__init__(no, **kw)
        self.comm = comm
        if self.is_diis:
            self.mixer.allreduce = comm.all_reduce_sum

    # ---- helpers ---------------------------------------------------------
    def _narrow(self, sub, name, t):
        """Restrict index 'a' of an operand to this rank's rows (pre-sharded blocks already are)."""
        if "a" not in sub:
            return t
        pos = sub.index("a")
        if name in SHARD_DIMS:
            if SHARD_DIMS[name] != pos:
                raise AssertionError("sharded block %s used with a on another index: %s" % (name, sub))
            return t
        return self.shard.rows(t, pos)

    def _eval_rows(self, coef, spec, names, src, out):
        """out (local rows along 'a') += coef * einsum(spec) with every operand restricted to A."""
        subs = spec.split("->")[0].split(",")
        ops = [self._narrow(s, n, src[n]) for s, n in zip(subs, names)]
        bk.einsum(spec, *ops, out=out, alpha=coef, beta=1.0)

    def _dressed_fock(self, fock, T1, dV, shared):
        """ccsd.py:226-288.  The four rows that read V_iabc (through the shared partial traces G3 /
        G4, local rows [na, v]) fill this rank's rows; the other rows read replicated o^2v^2 blocks
        and produce nP^2 numbers or fewer, so they are dealt out over the ranks term by term.  One
        all-reduce of an nP x nP matrix assembles both."""
        no, sh, comm = self.no, self.shard, self.comm
        src = dict(dV)
        src.update(t=T1, foo=fock[:no, :no], fvv=fock[no:, no:], fov=fock[:no, no:])
        src.update(shared)                                       # G3 / G4: [na, v]
        acc = bk.zeros(*fock.shape)
        views = {"ov": acc[:no, no:], "vo": acc[no:, :no], "oo": acc[:no, :no], "vv": acc[no:, no:]}
        a0, a1 = no + sh.lo, no + sh.lo + sh.na
        mine = {"vo": acc[a0:a1, :no], "vv": acc[a0:a1, no:]}
        turn = 0
        for blk, rows in FOCK_TERMS.items():
            for coef, spec, names in rows:
                names = names.split()
                if any(n in FOCK_SHARED for n in names):          # local rows in, local rows out
                    bk.einsum(spec, *[src[n] for n in names], out=mine[blk], alpha=coef, beta=1.0)
                    continue
                if turn % comm.size == comm.rank:
                    bk.einsum(spec, *[src[n] for n in names], out=views[blk], alpha=coef, beta=1.0)
                turn += 1
        comm.all_reduce_sum(acc)
        return bk.lincomb([1.0, 1.0], [fock.contiguous(), acc])

    def _singles_residual(self, ft, T1, T2, dV):
        """ccsd.py:423-438; the V_aibc term is evaluated on this rank's rows, the other terms (vo-sized
        results of reductions over the replicated amplitudes) are dealt out over the ranks."""
        no, sh, comm = self.no, self.shard, self.comm
        Tt = bk.tilde(T2, swap_ij=True)
        src = dict(dV)
        src.update(t=T1, Tt=Tt, fov=ft[:no, no:])
        acc = bk.zeros(T1.shape[0], no)
        turn = 0
        for coef, spec, names in SINGLES_TERMS:
            names = names.split()
            if "aibc" in names:
                self._eval_rows(coef, spec, names, src, sh.rows(acc, 0))
                continue
            if turn % comm.size == comm.rank:
                bk.einsum(spec, *[src[n] for n in names], out=acc, alpha=coef, beta=1.0)
            turn += 1
        comm.all_reduce_sum(acc)
        return bk.lincomb([1.0, 1.0], [bk.copy(ft[no:, :no]), acc])

    def _dressed_rows(self, key, T1, dV, a_dim, skip_tau=False, shared=None):
        """Local rows (a in A) of a T1-dressed block, returned with the a index FIRST
        ([na, ...other indices in their original order])."""
        sh = self.shard
        srcv = dV[key] if key in SHARD_DIMS else sh.rows(dV[key], a_dim)
        order = [a_dim] + [d for d in range(4) if d != a_dim]
        buf = bk.copy(srcv.permute(*order))                      # [na, ...], contiguous
        inv = [order.index(d) for d in range(4)]
        view = buf.permute(*inv)                                 # original index order, strided
        src = dict(dV)
        src["t"] = T1
        for coef, spec, source, is_tau in V_TERMS[key]:
            if skip_tau and is_tau:
                continue
            nt = spec.split("->")[0].count(",")
            if source in SHARED_PRODUCTS:                        # X3 / X4: local rows already
                bk.einsum(spec, shared[source], out=view, alpha=coef, beta=1.0)
                continue
            self._eval_rows(coef, spec, [source] + ["t"] * nt, src, view)
        return buf

    def _tau_ladder(self, T1, dV):
        """The folded particle-particle ladder of ccsd.tau_ladder on local rows."""
        sh = self.shard

        def apply(T2, R):
            ct = bk.contract_terms
            tau = bk.axpby(1.0, T2, 0.0, bk.empty_even_pitch(T2.shape[0], T2.shape[1], T2.shape[2]))
            ct("abij", [(1.0, "ai", T1, "bj", T1)], out=tau, beta=1.0)
            with bk.timed("pp_ladder"):
                ct("abij", [(1.0, "abcd", dV["abcd"], "cdij", tau)], out=R, beta=1.0)
            T1a = sh.rows(T1, 0)
            # W1[k,b,i,j] for b in A from the local V_iabc[:,A], gathered along b
            no = T1.shape[1]
            W1l, W2 = ccsd.pair_with_tau(dV["iabc"], dV["aibc"], tau, no)     # [k, b in A, i, j], [a in A, l, i, j]
            W1 = sh.gather_dim1(bk.copy(W1l.permute(1, 0, 2, 3)))             # rows first for the gather (o^3 v / N numbers)
            ct("abij", [(-1.0, "ak", T1a, "kbij", W1)], out=R, beta=1.0)
            # o^4 output, contraction over (c,d): each rank sums its c in A, then all-reduce
            W3 = sh.all_reduce(ct("klij", [(1.0, "klcd", sh.rows(dV["ijab"], 2), "cdij", sh.rows(tau, 0))]))
            ct("alij", [(-1.0, "ak", T1a, "klij", W3)], out=W2, beta=1.0)
            ct("abij", [(-1.0, "bl", T1, "alij", W2)], out=R, beta=1.0)
        return apply

    # ---- driver ----------------------------------------------------------
    def setup(self, t_fock_pq, dict_blocks, level_shift=0., amps=None):
        no = self.no
        fock_host = bk.tonumpy(t_fock_pq)
        nv = fock_host.shape[0] - no
        self.shard = Shard(self.comm, nv)
        if not isinstance(dict_blocks, dict):
            # the reference call surface: a dense V_pqrs (numpy / tensor) that every rank holds;
            # each rank keeps views of its row blocks
            from .integral.partition import part_2_body_int
            dict_blocks = shard_blocks(part_2_body_int(no, bk.asdev(dict_blocks)), self.shard)
        self.local_rows = self.shard.na
        st = self._st = {}
        st["want_numpy"] = False
        st["eps_i"] = bk.asdev(fock_host.diagonal()[:no].copy())
        st["eps_a"] = bk.asdev(fock_host.diagonal()[no:].copy())
        st["fock"] = bk.asdev(fock_host)
        st["dV"] = {k: (bk.asdev(v) if v is not None else None) for k, v in dict_blocks.items()}
        for k, dim in SHARD_DIMS.items():
            if st["dV"][k].shape[dim] != self.shard.na:
                raise ValueError("block %s must be the local row block (%d rows)" % (k, self.shard.na))
        st["dtype_name"] = "float64"
        st["shift"] = level_shift
        e_mp2, T2 = mp2.solve_device(st["eps_i"], st["eps_a"], st["dV"]["ijab"], st["dV"]["abij"], level_shift)
        # the exchanges (all-gather, row transpose) do not carry momentum rules yet: a sharded sweep
        # starts from untagged amplitudes and keeps the dense ring products
        bk.drop_momentum(T2)
        T1 = bk.zeros(nv, no)
        if amps is not None:
            T1, T2 = bk.asdev(amps[0]).contiguous(), bk.asdev(amps[1]).contiguous()
        st["T1"], st["T2"] = T1, T2
        st["amps_host"] = None
        st["scal"] = bk.zeros(8)
        st["e_mp2"] = e_mp2
        st["iteration"] = 0
        st["V_ijab_e"] = ccsd.energy_layout(st["dV"]["ijab"])
        return e_mp2

    def sweep(self):
        st, sh = self._st, self.shard
        no, dV, fock = self.no, st["dV"], st["fock"]
        T1, T2, scal = st["T1"], st["T2"], st["scal"]
        eps_i, eps_a, shift = st["eps_i"], st["eps_a"], st["shift"]
        rows = (sh.lo, sh.na)
        st["iteration"] += 1
        shared = ccsd.t1_shared(T1, dV)            # X3 / X4 / G3 / G4 on the local rows of V_iabc[:,A]
        ft = self._dressed_fock(fock, T1, dV, shared)
        R1 = self._singles_residual(ft, T1, T2, dV)
        V_abij = self._dressed_rows("abij", T1, dV, 0, skip_tau=True)                 # [A,b,i,j]
        # local rows [A,i,j,b] -> full [i,a,j,b] views; the two all-gathers travel while the ladder runs
        dim1 = lambda t: t.transpose(0, 1)
        V_iajb = sh.gather_async(self._dressed_rows("iajb", T1, dV, 1, shared=shared), view=dim1)
        V_iabj = sh.gather_async(self._dressed_rows("iabj", T1, dV, 1, shared=shared), view=dim1)
        del shared
        R2 = ccd.doubles_residual(no, ft, T2, ccsd.dressed_block("klij", T1, dV), dV["ijab"], V_abij, V_iajb,
                                  V_iabj, None, is_dcd=self.is_dcd, pp_ladder=self._tau_ladder(T1, dV),
                                  shard=sh)
        del V_abij, V_iajb, V_iabj
        dT1 = bk.update_singles(eps_i, eps_a, shift, self.delta, R1, T1)
        T2l = sh.rows(T2, 0).clone()
        dT2 = bk.update_doubles(eps_i, eps_a, shift, self.delta, R2, T2l, scal[3:4], rows=rows)
        del R1, R2
        if self.is_diis:
            T1, T2l = self.mixer.mix([dT1, dT2], [T1, T2l], sharded=[False, True])
        T2 = sh.gather_async(T2l)                   # ... while the energy of the local rows is summed
        bk.energy_doubles(T2l, st["V_ijab_e"], scal, T1=T1, rows=rows)
        T2 = T2.wait_result()
        st["T1"], st["T2"] = T1, T2
        self.comm.all_reduce_sum(scal[0:4])
        bk.contract_terms("", [(2.0, "ia", fock[:no, no:], "ai", T1)], out=scal[4])
        s = scal.cpu().numpy()
        return float(s[4]), float(s[0]), float(s[1]), float(np.sqrt(s[2])), float(np.sqrt(s[3]))

    def sweep_host(self, t1_host, t2_host):
        """Host-buffer form: ``t2_host`` is this rank's ROW BLOCK of T2 in (pinned) host memory,
        ``t1_host`` the full T1; the new amplitudes are written back into them."""
        st, sh = self._st, self.shard
        t1 = t1_host if isinstance(t1_host, torch.Tensor) else torch.from_numpy(t1_host)
        t2 = t2_host if isinstance(t2_host, torch.Tensor) else torch.from_numpy(t2_host)
        st["T1"] = t1.to(bk.device(), non_blocking=True)
        st["T2"] = sh.gather(t2.to(bk.device(), non_blocking=True))
        out = self.sweep()
        t1.copy_(st["T1"], non_blocking=True)
        t2.copy_(sh.rows(st["T2"], 0), non_blocking=True)
        if torch.cuda.is_available():
            torch.cuda.current_stream().synchronize()
        return out
