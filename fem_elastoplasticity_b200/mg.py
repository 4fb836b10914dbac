"""Geometric multigrid preconditioned CG on the device (kernels in csrc/mg.cu, C ABI in include/fem_b200.h).

The reference solves every Newton system with a dense LU (Plasticity2D_DP/pythonFEM.py:1062-1066); on the meshes this
package targets that is replaced by CG.  Point-Jacobi needs O(N) iterations (57 500 at 16M elements), the two-level method
(twolevel.py) ~1 900; a V-cycle with Chebyshev-Jacobi smoothing brings the count to ~30-50 independent of the mesh size.
Any SPD preconditioner yields the reference's solution, so parity is unaffected.

Applies to meshes whose nodes lie on a uniform lattice with edges no longer than one lattice step (the uniform P1/Q1
meshes of the footing problem and of configs 1/4/5); ``MultigridPCG`` raises ``MultigridUnsupported`` otherwise and the
caller keeps the two-level / Jacobi solver (the unstructured tsx mesh has 952 unknowns).

This module only computes layouts, owns the buffers and sequences kernel launches; PyTorch supplies device memory, the
set-up collectives and the dense factorisation of the coarsest level (set-up only)."""
import ctypes as C
import time

import torch

from ._lib import call, load
from .plan import _ptr, _stream

MAX_LEVELS, MAX_DEGREE, MAX_PEERS = 16, 8, 16


class MultigridUnsupported(ValueError):
    pass


class Exchange(C.Structure):
    _fields_ = [("n_send", C.c_int32), ("n_wait", C.c_int32), ("src_off", C.c_int64 * MAX_PEERS), ("count", C.c_int64 * MAX_PEERS),
                ("dst", C.c_void_p * MAX_PEERS), ("dst_flag", C.c_void_p * MAX_PEERS), ("wait_flag", C.c_void_p * MAX_PEERS),
                ("seq", C.c_void_p)]


class Level(C.Structure):
    _fields_ = [("nxn", C.c_int32), ("nrows", C.c_int32), ("g0", C.c_int32), ("own_lo", C.c_int32), ("own_hi", C.c_int32),
                ("nrows_global", C.c_int32), ("res_lo", C.c_int32), ("res_hi", C.c_int32),
                ("S", C.c_void_p), ("S32", C.c_void_p), ("dinv", C.c_void_p), ("b", C.c_void_p), ("xa", C.c_void_p), ("xb", C.c_void_p), ("d", C.c_void_p),
                ("r", C.c_void_p), ("c1", C.c_double * MAX_DEGREE), ("c2", C.c_double * MAX_DEGREE),
                ("ex_xa", Exchange), ("ex_xb", Exchange), ("ex_r", Exchange), ("ex_b", Exchange)]


class Desc(C.Structure):
    _fields_ = [("n_levels", C.c_int32), ("degree", C.c_int32), ("LX", C.c_int32), ("lat_rows", C.c_int32), ("g0", C.c_int32),
                ("nrows_global", C.c_int32), ("lat", C.c_void_p), ("node_lat", C.c_void_p), ("own_node_lo", C.c_int64),
                ("own_node_hi", C.c_int64), ("mask", C.c_void_p), ("dinv", C.c_void_p), ("xa", C.c_void_p), ("xb", C.c_void_p),
                ("d", C.c_void_p), ("r", C.c_void_p), ("c1", C.c_double * MAX_DEGREE), ("c2", C.c_double * MAX_DEGREE),
                ("ex_xa", Exchange), ("ex_xb", Exchange), ("ex_r", Exchange), ("lev", Level * MAX_LEVELS), ("coarse_inv", C.c_void_p),
                ("K32", C.c_void_p), ("err", C.c_void_p), ("lat32", C.c_void_p), ("lat32_stride", C.c_int64), ("lat32_nw", C.c_int32),
                ("lat32_pad", C.c_int32)]


def chebyshev_coefficients(lmax, ratio, degree):
    """d_k = c1[k] d_{k-1} + c2[k] D^-1 r_k, x_{k+1} = x_k + d_k: the Chebyshev polynomial for the interval
    [lmax/ratio, lmax] of D^-1 A."""
    lmin = lmax / ratio
    theta, delta = 0.5 * (lmax + lmin), 0.5 * (lmax - lmin)
    sigma = theta / delta
    rho = 1.0 / sigma
    c1, c2 = [0.0], [1.0 / theta]
    for _ in range(1, degree):
        rho_new = 1.0 / (2.0 * sigma - rho)
        c1.append(rho_new * rho)
        c2.append(2.0 * rho_new / delta)
        rho = rho_new
    return c1, c2


def check_schedule(hint, check_every):
    """First iteration at which a solve looks at its residual, given the iteration count ``hint`` of the previous solve with
    the same tolerance (None: no previous solve): four iterations before it, rounded down to a multiple of ``check_every``."""
    return 0 if hint is None else max(0, ((hint - 4) // check_every) * check_every)


def next_check(it, n_it, check_every, skip_until):
    """Iteration index of the next convergence check after iteration ``it``."""
    return min(n_it, max((it // check_every + 1) * check_every, skip_until))


def level_layouts(LX, NY, owned, max_coarse_dofs=2500, min_owned_rows=3, max_levels=MAX_LEVELS, replicate_below=600000):
    """Layouts of the structured levels l = 1 .. L over an LX x NY node lattice whose rows are owned by the ranks as the
    half-open global ranges ``owned`` (one per rank, ascending, covering [0, NY)).

    Level l+1 keeps every second lattice point of level l (ceil: an odd cell count adds one coarse node row/column beyond
    the last fine one).  Coarse row J belongs to the owner of fine row 2J (the last rank takes the extra row).  A level is
    DISTRIBUTED while every rank owns at least ``min_owned_rows`` rows and the level has more than ``replicate_below`` nodes
    (smaller levels: a sweep over the WHOLE level costs < 20 us, its share on one rank ~10 us, and each of the ~6 exchanges
    per level and V-cycle ~13 us - computing the level redundantly is cheaper than exchanging.  Measured on two B200s,
    32M elements: 50 000 -> 3.26 ms per CG iteration, 300 000 / 600 000 -> 3.16 ms, 1 200 000 -> 3.25 ms): its local arrays hold the owned rows plus one ghost row on each side that exists.  Below that, and always on
    the last (densely solved) level, the level is REPLICATED:
    every rank holds all rows; on the first replicated level a rank restricts only its share ``res`` of the rows and the
    shares are gathered.  Returns a list of dicts: nxn, nrows_global, replicated, ranks = [(g0, nrows, own_lo, own_hi,
    res_lo, res_hi)] in local row indices."""
    world = len(owned)
    assert owned[0][0] == 0 and owned[-1][1] == NY and all(owned[i][1] == owned[i + 1][0] for i in range(world - 1)), owned
    levels, nxn, N, own, replicated = [], LX, NY, list(owned), world == 1
    while True:
        nxn_c, N_c = -(-(nxn - 1) // 2) + 1, -(-(N - 1) // 2) + 1
        share = [(-(-lo // 2), N_c if hi == N else -(-hi // 2)) for lo, hi in own]
        last = 2 * nxn_c * N_c <= max_coarse_dofs or len(levels) == max_levels - 1 or (nxn_c <= 2 and N_c <= 2)
        rep = replicated or last or min(hi - lo for lo, hi in share) < min_owned_rows or nxn_c * N_c <= replicate_below
        ranks = []
        for lo, hi in share:
            if rep:
                res = (0, N_c) if replicated else (lo, hi)
                ranks.append((0, N_c, 0, N_c, res[0], res[1]))
            else:
                g0, end = max(0, lo - 1), min(N_c, hi + 1)
                ranks.append((g0, end - g0, lo - g0, hi - g0, lo - g0, hi - g0))
        levels.append({"nxn": nxn_c, "nrows_global": N_c, "replicated": rep, "first_replicated": rep and not replicated, "ranks": ranks,
                       "owned_global": share})
        if last:
            return levels
        nxn, N, replicated = nxn_c, N_c, rep
        own = [(0, N_c)] * world if rep else share


def infer_lattice(coord):
    """(x0, y0, hx, hy, LX, NY) of the uniform lattice the (2, n_n) device coordinates lie on (checked later, node by node,
    by fem_mg_lattice)."""
    x, y = coord[0], coord[1]
    x0, x1, y0, y1 = float(x.min()), float(x.max()), float(y.min()), float(y.max())

    def step(v, lo):
        d = v - lo
        pos = d[d > 1e-9 * max(abs(lo), float(d.max()), 1e-300)]
        return float(pos.min()) if pos.numel() else 1.0
    hx, hy = step(x, x0), step(y, y0)
    return x0, y0, hx, hy, int(round((x1 - x0) / hx)) + 1, int(round((y1 - y0) / hy)) + 1


def check_abi():
    """The ctypes structures above against the library's own sizeof."""
    lib = load()
    got = tuple(int(lib.fem_mg_sizeof(i)) for i in range(3))
    want = (C.sizeof(Exchange), C.sizeof(Level), C.sizeof(Desc))
    if got != want:
        raise ImportError(f"fem_mg_* structure layout mismatch: library {got}, binding {want}")


class MultigridPCG:
    """CG preconditioned by one V-cycle per iteration.  ``mask``: unknowns of this rank (free; free AND owned on a strip
    partition); ``free_mask``: all free DOFs of the local vectors (ghost rows included).  ``setup(k_vals)`` builds the coarse
    operators (Galerkin) from ``k_vals`` - for the Newton loop the elastic matrix, kept for every tangent solve: level 0
    always uses the matrix being solved.  ``solve`` mirrors TwoLevelPCG.solve."""

    def __init__(self, plan, mask, part=None, free_mask=None, degree=2, ratio=16.0, max_coarse_dofs=2500, lattice=None, use_graph=True,
                 smoother_f32=True, replicate_below=600000):
        check_abi()
        self.plan, self.mask = plan, mask
        self.part = part if (part is not None and part.world > 1) else None
        self.free_mask = free_mask if free_mask is not None else mask
        if self.part is not None and free_mask is None:
            raise ValueError("MultigridPCG on a partition needs free_mask (free DOFs including ghost rows)")
        if not 1 <= degree <= MAX_DEGREE:
            raise ValueError("degree")
        self.degree, self.ratio, self.use_graph = degree, ratio, use_graph
        # FP32 copy of the matrix for the level-0 smoother / residual of the V-cycle (the CG itself stays on the FP64 matrix)
        self.k32 = torch.zeros(plan.nnz, dtype=torch.float32, device=plan.device) if smoother_f32 else None
        self.device = dev = plan.device
        n = plan.n_dof
        z = lambda m, dt=torch.float64: torch.zeros(m, dtype=dt, device=dev)  # noqa: E731
        # ---- level 0 lattice
        world, rank = (self.part.world, self.part.rank) if self.part is not None else (1, 0)
        self.world, self.rank = world, rank
        if lattice is None:
            if self.part is not None:
                p = self.part
                lattice = (0.0, 0.0, p.size_x / p.nx, p.size_y / p.ny_global, p.nx + 1, p.ny_global + 1)
            else:
                lattice = infer_lattice(plan.coord)
        x0, y0, hx, hy, LX, NY = lattice
        if self.part is not None:
            p = self.part
            g0, lat_rows = p.iy0, p.n_node_rows
            owned = [(0 if r == 0 else r * p.ny_loc + 1, (r + 1) * p.ny_loc + 1) for r in range(world)]
        else:
            g0, lat_rows, owned = 0, NY, [(0, NY)]
        if LX * lat_rows > 4 * plan.n_n + 64:
            raise MultigridUnsupported(f"mesh does not fill a uniform lattice ({LX} x {lat_rows} points for {plan.n_n} nodes)")
        self.lattice, self.g0, self.lat_rows, self.owned = (x0, y0, hx, hy, LX, NY), g0, lat_rows, owned
        self.lat, self.node_lat, err = z(LX * lat_rows, torch.int32), z(plan.n_n, torch.int32), z(1, torch.int32)
        call("fem_mg_lattice", plan.n_n, _ptr(plan.coord), x0, y0, hx, hy, LX, lat_rows, g0, _ptr(self.lat), _ptr(self.node_lat), _ptr(err), _stream())
        if int(err.item()) != 0:
            raise MultigridUnsupported(f"mesh nodes are not on a uniform lattice (code {int(err.item())})")
        own_rows = (owned[rank][0] - g0, owned[rank][1] - g0)
        if self.part is not None:   # ghost rows are refreshed by row copies: nodes must be numbered along the lattice
            if not bool((self.node_lat == torch.arange(plan.n_n, dtype=torch.int32, device=dev)).all()):
                raise MultigridUnsupported("partitioned multigrid needs lattice-ordered node numbering")
        self.own_nodes = (own_rows[0] * LX, own_rows[1] * LX) if self.part is not None else (0, plan.n_n)
        self._lattice_stencil(LX, lat_rows)
        self.layouts = level_layouts(LX, NY, owned, max_coarse_dofs=max_coarse_dofs, replicate_below=replicate_below)
        self.n_levels = len(self.layouts)
        # ---- buffers (on a partition the vectors whose ghost rows travel live in one symmetric-memory arena)
        self._arena_slots, self._ex_ids = {}, {}
        if self.part is not None:
            self._make_arena(n)
        a = self._vec
        self.r, self.q, self.x, self.z = (z(n) for _ in range(4))
        self.minv = z(2 * n)                              # inverse 2x2 diagonal blocks of the matrix being solved, two planes
        self.p = a("p", n)
        self.scal = z(8)
        self.v0 = {"xa": a("xa0", n), "xb": a("xb0", n), "d": z(n), "r": a("r0", n)}
        self.lv = []
        for li, lay in enumerate(self.layouts):
            g0l, nrows, own_lo, own_hi, res_lo, res_hi = lay["ranks"][rank]
            nn = lay["nxn"] * nrows
            self.lv.append({"nxn": lay["nxn"], "nrows": nrows, "g0": g0l, "own": (own_lo, own_hi), "res": (res_lo, res_hi), "n": nn,
                            "N": lay["nrows_global"], "rep": lay["replicated"], "first_rep": lay["first_replicated"],
                            "S": z(36 * nn), "dinv": z(4 * nn), "d": z(2 * nn), "b": a(f"b{li + 1}", 2 * nn),
                            "xa": a(f"xa{li + 1}", 2 * nn), "xb": a(f"xb{li + 1}", 2 * nn), "r": a(f"r{li + 1}", 2 * nn), "lmax": None})
        self.coarse_inv, self.desc, self.setup_seconds, self.lmax0 = None, None, None, None
        self._graph, self._graph_key = None, None
        self.launches_last = 0

    def _lattice_stencil(self, LX, lat_rows):
        """Level 0 as a 7-point stencil (fem_mg_fine_lattice): the FP32 smoother on one GPU, node id == lattice point, every
        neighbour inside the 3x3 window and one diagonal orientation.  Otherwise (and on strip partitions, where the stencil
        has not been checked against the ghost rows) the smoother keeps the block-CSR copy."""
        self.k32s, self.lat32_stride, self.lat32_nw = None, 0, 0
        P = self.plan
        if self.k32 is None or self.part is not None or LX * lat_rows != P.n_n:
            return
        err = torch.zeros(1, dtype=torch.int32, device=self.device)
        call("fem_mg_lattice_check", P._h, _ptr(self.node_lat), LX, _ptr(err), _stream())
        e = int(err.item())
        if e & 3 or e == 12:
            return
        self.lat32_nw = 1 if e == 8 else 0
        self.lat32_stride = (P.n_n + 31) // 32 * 32                # every plane starts on a 128-byte line
        self.k32s = torch.zeros(16 * self.lat32_stride, dtype=torch.float32, device=self.device)

    @property
    def fine_lattice(self):
        return self.k32s is not None

    def to_f32(self, k_vals):
        """The FP32 copies the level-0 smoother reads: the block-CSR copy k32 and, when level 0 runs on the lattice, the
        stencil planes k32s (one pass over k_vals)."""
        if self.k32s is not None:
            call("fem_mg_to_f32_lattice", self.plan._h, _ptr(k_vals), _ptr(self.k32), _ptr(self.k32s), self.lat32_stride, self.lattice[4],
                 self.lat32_nw, _stream())
        elif self.k32 is not None:
            call("fem_mg_to_f32", self.plan.nnz, _ptr(k_vals), _ptr(self.k32), _stream())

    # -- multi-GPU plumbing (set-up collectives through torch.distributed; the solve uses fem_mg_exchange) ----------------
    def _vec(self, name, size):
        """A zeroed vector; the arena slot ``name`` when this vector is exchanged between ranks."""
        if name in self._arena_slots:
            off, _ = self._arena_slots[name]
            return self.arena[off:off + size]
        return torch.zeros(size, dtype=torch.float64, device=self.device)

    def _make_arena(self, n):
        """One symmetric allocation (CUDA IPC mappings over NVLink) for every exchanged vector, the same offsets on every
        rank, and the communication block: per exchange 16 flag words (one per source rank) + sequence number + ticket,
        the sticky time-out word, and the lines of the scalar all-reduce."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        dev, world = self.device, self.world
        nmax = torch.tensor([n], dtype=torch.int64, device=dev)
        dist.all_reduce(nmax, op=dist.ReduceOp.MAX)
        slots = [("p", int(nmax.item())), ("xa0", int(nmax.item())), ("xb0", int(nmax.item())), ("r0", int(nmax.item()))]
        for li, lay in enumerate(self.layouts):
            if not lay["replicated"]:
                sz = max(2 * lay["nxn"] * rk[1] for rk in lay["ranks"])
                slots += [(f"xa{li + 1}", sz), (f"xb{li + 1}", sz), (f"r{li + 1}", sz)]
            elif lay["first_replicated"]:
                slots += [(f"b{li + 1}", 2 * lay["nxn"] * lay["nrows_global"])]
        off = 0
        for name, sz in slots:
            self._arena_slots[name] = (off, sz)
            self._ex_ids[name] = len(self._ex_ids)
            off += sz + (sz & 1)
        self.arena = symm.empty(off, dtype=torch.float64, device=dev)
        self.arena.zero_()
        self._arena_hdl = symm.rendezvous(self.arena, dist.group.WORLD)
        self._arena_peers = [self.arena.data_ptr() if r == self.rank else self._arena_hdl.get_buffer(r, (off,), torch.float64).data_ptr() for r in range(world)]
        n_ex = len(self._ex_ids)
        self.W_SEQ = n_ex * MAX_PEERS
        self.W_ERR = self.W_SEQ + 2 * n_ex
        self.W_ARSEQ = self.W_ERR + 1
        self.W_LINES = self.W_ARSEQ + 1
        n_words = self.W_LINES + 512
        self.comm = symm.empty(n_words, dtype=torch.int64, device=dev)
        self.comm.zero_()
        self._comm_hdl = symm.rendezvous(self.comm, dist.group.WORLD)
        self._comm_views = [self.comm if r == self.rank else self._comm_hdl.get_buffer(r, (n_words,), torch.int64) for r in range(world)]
        self._comm_peers = [v.data_ptr() for v in self._comm_views]
        self._comm_table = (C.c_void_p * world)(*self._comm_peers)
        torch.cuda.synchronize()
        self._comm_hdl.barrier(channel=0)                # every arena and block is zeroed before any peer may store into it
        torch.cuda.synchronize()

    def _halo_desc(self, name, width, rank_rows):
        """Exchange of the two boundary rows of vector ``name`` (rows of ``width`` nodes) with the neighbouring strips;
        rank_rows[r] = (g0, nrows, own_lo, own_hi) of every rank."""
        ex = Exchange()
        if self.part is None or name not in self._ex_ids:
            return ex
        e, (off, _), rk = self._ex_ids[name], self._arena_slots[name], self.rank
        g0, nrows, lo, hi = rank_rows[rk]
        k = 0
        for nb, src_row, exists in ((rk + 1, hi - 1, hi < nrows), (rk - 1, lo, lo > 0)):
            if not exists:
                continue
            dst_row = g0 + src_row - rank_rows[nb][0]
            assert 0 <= dst_row < rank_rows[nb][1] and not rank_rows[nb][2] <= dst_row < rank_rows[nb][3], (name, rk, nb, dst_row)
            ex.src_off[k], ex.count[k] = src_row * width, width
            ex.dst[k] = self._arena_peers[nb] + 8 * off + 16 * dst_row * width
            ex.dst_flag[k] = self._comm_peers[nb] + 8 * (e * MAX_PEERS + rk)
            ex.wait_flag[k] = self._comm_peers[rk] + 8 * (e * MAX_PEERS + nb)
            k += 1
        ex.n_send = ex.n_wait = k
        ex.seq = self._comm_peers[rk] + 8 * (self.W_SEQ + 2 * e)
        return ex

    def _gather_desc(self, name, width, res):
        """Every rank's share of the rows of ``name`` (first replicated level) to every other rank."""
        ex = Exchange()
        if self.part is None or name not in self._ex_ids:
            return ex
        e, (off, _), rk = self._ex_ids[name], self._arena_slots[name], self.rank
        k = 0
        for r in range(self.world):
            if r == rk:
                continue
            ex.src_off[k], ex.count[k] = res[0] * width, (res[1] - res[0]) * width
            ex.dst[k] = self._arena_peers[r] + 8 * off + 16 * res[0] * width
            ex.dst_flag[k] = self._comm_peers[r] + 8 * (e * MAX_PEERS + rk)
            ex.wait_flag[k] = self._comm_peers[rk] + 8 * (e * MAX_PEERS + r)
            k += 1
        ex.n_send = ex.n_wait = k
        ex.seq = self._comm_peers[rk] + 8 * (self.W_SEQ + 2 * e)
        return ex

    def _halo_rows(self, lv, t):
        """Forward halo of a level array viewed as (planes, nrows, width): ghost rows <- the neighbours' boundary rows."""
        import torch.distributed as dist
        lo, hi = lv["own"]
        ops, tmp = [], []
        if lo > 0:          # lower neighbour exists
            s, rcv = t[:, lo, :].contiguous(), torch.empty_like(t[:, lo - 1, :].contiguous())
            ops += [dist.P2POp(dist.isend, s, self.rank - 1), dist.P2POp(dist.irecv, rcv, self.rank - 1)]
            tmp.append((lo - 1, rcv))
        if hi < lv["nrows"]:
            s, rcv = t[:, hi - 1, :].contiguous(), torch.empty_like(t[:, hi, :].contiguous())
            ops += [dist.P2POp(dist.isend, s, self.rank + 1), dist.P2POp(dist.irecv, rcv, self.rank + 1)]
            tmp.append((hi, rcv))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        for row, rcv in tmp:
            t[:, row, :] = rcv

    def _halo_add_rows(self, lv, t):
        """Reverse halo: the partial sums a rank scattered into its ghost rows are added to the owners' rows."""
        import torch.distributed as dist
        lo, hi = lv["own"]
        ops, tmp = [], []
        if lo > 0:
            s, rcv = t[:, lo - 1, :].contiguous(), torch.empty_like(t[:, lo, :].contiguous())
            ops += [dist.P2POp(dist.isend, s, self.rank - 1), dist.P2POp(dist.irecv, rcv, self.rank - 1)]
            tmp.append((lo, rcv))
        if hi < lv["nrows"]:
            s, rcv = t[:, hi, :].contiguous(), torch.empty_like(t[:, hi - 1, :].contiguous())
            ops += [dist.P2POp(dist.isend, s, self.rank + 1), dist.P2POp(dist.irecv, rcv, self.rank + 1)]
            tmp.append((hi - 1, rcv))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        for row, rcv in tmp:
            t[:, row, :] += rcv

    def _all_reduce(self, t, op=None):
        if self.part is not None:
            import torch.distributed as dist
            dist.all_reduce(t, op=op if op is not None else dist.ReduceOp.SUM)

    # -- set-up ---------------------------------------------------------------------------------------------------------
    def setup(self, k_vals):
        """Coarse operators A_{l+1} = P^T A_l P of ``k_vals``, inverse diagonals, eigenvalue bounds of D^-1 A on every level,
        dense inverse of the last level."""
        import torch.distributed as dist
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        P, dev = self.plan, self.device
        x0, y0, hx, hy, LX, NY = self.lattice
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        # level 1 from the block-CSR matrix: rows of this rank's unknowns x all free columns
        l1 = self.lv[0]
        call("fem_mg_galerkin_fine", P._h, _ptr(k_vals), _ptr(self.mask), _ptr(self.free_mask), _ptr(self.lat), self.lat_rows, _ptr(self.node_lat),
             LX, self.g0, l1["nxn"], l1["nrows"], l1["g0"], _ptr(l1["S"]), _ptr(err), _stream())
        if int(err.item()) != 0:
            raise MultigridUnsupported(f"mesh edges do not fit the 9-point coarse stencil (code {int(err.item())})")
        if self.part is not None:
            s3 = l1["S"].view(36, l1["nrows"], l1["nxn"])
            if l1["rep"]:
                dist.all_reduce(l1["S"])
            else:
                self._halo_add_rows(l1, s3)
                self._halo_rows(l1, s3)
        for li in range(1, self.n_levels):
            f, c = self.lv[li - 1], self.lv[li]
            rows = c["res"] if c["first_rep"] else c["own"]
            call("fem_mg_galerkin_stencil", f["nxn"], f["nrows"], f["g0"], f["N"], _ptr(f["S"]), c["nxn"], c["nrows"], c["g0"], rows[0], rows[1],
                 _ptr(c["S"]), _stream())
            if self.part is not None:
                if c["first_rep"]:
                    dist.all_reduce(c["S"])                  # rows outside the share are zero
                elif not c["rep"]:
                    self._halo_rows(c, c["S"].view(36, c["nrows"], c["nxn"]))
        for lv in self.lv:
            nn = lv["n"]
            dmax = torch.maximum(lv["S"][16 * nn:17 * nn].max(), lv["S"][19 * nn:20 * nn].max()).reshape(1)
            self._all_reduce(dmax, op=None if self.part is None else dist.ReduceOp.MAX)
            call("fem_mg_level_finalize", nn, _ptr(lv["S"]), 1e-14 * float(dmax.item()), _ptr(lv["dinv"]), _stream())
        # eigenvalue bounds (power iteration on D^-1 A), Chebyshev coefficients
        self.lmax0 = 1.1 * self._power_fine(k_vals)
        for lv in self.lv[:-1]:
            lv["lmax"] = 1.1 * self._power_level(lv)
        # dense inverse of the last level
        last = self.lv[-1]
        nc = 2 * last["n"]
        A = torch.empty((nc, nc), dtype=torch.float64, device=dev)
        call("fem_mg_stencil_to_dense", last["nxn"], last["nrows"], _ptr(last["S"]), _ptr(A), _stream())
        A = 0.5 * (A + A.t())
        self.coarse_inv = torch.cholesky_inverse(torch.linalg.cholesky(A)).contiguous()
        v = torch.randn((nc, 4), dtype=torch.float64, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
        self.inverse_residual = float(((A @ (self.coarse_inv @ v)) - v).norm() / v.norm())
        if not self.inverse_residual <= 1e-6:
            raise ArithmeticError(f"multigrid: dense inverse of the coarsest operator is inaccurate (residual {self.inverse_residual:.2e})")
        del A
        self._build_desc()
        torch.cuda.synchronize()
        self.setup_seconds = time.perf_counter() - t0
        return self

    @staticmethod
    def block_apply(dinv, v):
        """D^-1 v for the two-plane block inverse ``dinv`` (planes A = (i00, i01), B = (i01, i11) per node)."""
        n = v.numel()
        a, b, v2 = dinv[:n].view(-1, 2), dinv[n:2 * n].view(-1, 2), v.view(-1, 2)
        return torch.stack([a[:, 0] * v2[:, 0] + a[:, 1] * v2[:, 1], b[:, 0] * v2[:, 0] + b[:, 1] * v2[:, 1]], dim=1).reshape(-1)

    def block_jacobi(self, k_vals, out=None):
        out = self.minv if out is None else out
        call("fem_mg_block_jacobi", self.plan._h, _ptr(k_vals), _ptr(self.mask), _ptr(out), _stream())
        return out

    def _power_fine(self, k_vals, iters=20):
        P = self.plan
        dinv = self.block_jacobi(k_vals)
        g = torch.Generator(device=self.device).manual_seed(11 + self.rank)
        v = torch.randn(P.n_dof, dtype=torch.float64, device=self.device, generator=g) * self.mask
        y = torch.empty_like(v)
        lam = 1.0
        for _ in range(iters):
            if self.part is not None:
                self.part.halo_exchange(v)
            P.spmv(k_vals, v, mask=self.mask, out=y)
            y = self.block_apply(dinv, y)
            nrm = y.square().sum().reshape(1)
            self._all_reduce(nrm)
            lam = float(nrm.sqrt().item())
            v = y / lam
        return lam

    def _power_level(self, lv, iters=20):
        nn, (lo, hi) = lv["n"], lv["own"]
        g = torch.Generator(device=self.device).manual_seed(13 if lv["rep"] else 13 + self.rank)
        v = torch.zeros(2 * nn, dtype=torch.float64, device=self.device)
        w = lv["nxn"] * 2
        v[lo * w:hi * w] = torch.randn((hi - lo) * w, dtype=torch.float64, device=self.device, generator=g)
        y = torch.zeros_like(v)
        lam = 1.0
        for _ in range(iters):
            if self.part is not None and not lv["rep"]:
                self._halo_rows(lv, v.view(1, lv["nrows"], w))
            call("fem_mg_stencil_apply", lv["nxn"], lv["nrows"], lo, hi, _ptr(lv["S"]), _ptr(v), _ptr(y), _stream())
            y = self.block_apply(lv["dinv"], y)
            nrm = y[lo * w:hi * w].square().sum().reshape(1)
            if not lv["rep"]:
                self._all_reduce(nrm)
            lam = float(nrm.sqrt().item())
            v = y / lam
        return lam

    def _build_desc(self):
        d = Desc()
        x0, y0, hx, hy, LX, NY = self.lattice
        d.n_levels, d.degree, d.LX, d.lat_rows, d.g0, d.nrows_global = self.n_levels, self.degree, LX, self.lat_rows, self.g0, NY
        d.lat, d.node_lat = self.lat.data_ptr(), self.node_lat.data_ptr()
        d.own_node_lo, d.own_node_hi = self.own_nodes
        d.mask, d.dinv = self.mask.data_ptr(), self.minv.data_ptr()
        d.xa, d.xb, d.d, d.r = (self.v0[k].data_ptr() for k in ("xa", "xb", "d", "r"))
        c1, c2 = chebyshev_coefficients(self.lmax0, self.ratio, self.degree)
        for k in range(self.degree):
            d.c1[k], d.c2[k] = c1[k], c2[k]
        for li, lv in enumerate(self.lv):
            L = d.lev[li]
            L.nxn, L.nrows, L.g0, L.own_lo, L.own_hi, L.nrows_global = lv["nxn"], lv["nrows"], lv["g0"], lv["own"][0], lv["own"][1], lv["N"]
            L.res_lo, L.res_hi = lv["res"]
            L.S, L.dinv = lv["S"].data_ptr(), lv["dinv"].data_ptr()
            if self.k32 is not None and li < self.n_levels - 1:     # FP32 copy of the stencil for the smoother (as on level 0)
                lv["S32"] = lv["S"].to(torch.float32)
                L.S32 = lv["S32"].data_ptr()
            L.b, L.xa, L.xb, L.d, L.r = (lv[k].data_ptr() for k in ("b", "xa", "xb", "d", "r"))
            if lv["lmax"] is not None:
                c1, c2 = chebyshev_coefficients(lv["lmax"], self.ratio, self.degree)
                for k in range(self.degree):
                    L.c1[k], L.c2[k] = c1[k], c2[k]
        d.coarse_inv = self.coarse_inv.data_ptr()
        d.K32 = self.k32.data_ptr() if self.k32 is not None else 0
        d.err = 0
        if self.k32s is not None:
            d.lat32, d.lat32_stride, d.lat32_nw = self.k32s.data_ptr(), self.lat32_stride, self.lat32_nw
        self._fill_exchanges(d)
        self.desc = d

    def _fill_exchanges(self, d):
        if self.part is None:
            return
        p, LX = self.part, self.lattice[4]
        rows0 = [(r * p.ny_loc, p.ny_loc + 1 + (1 if r < self.world - 1 else 0), 1 if r > 0 else 0, p.ny_loc + 1) for r in range(self.world)]
        d.ex_xa, d.ex_xb, d.ex_r = (self._halo_desc(k, LX, rows0) for k in ("xa0", "xb0", "r0"))
        self.ex_p = self._halo_desc("p", LX, rows0)
        for li, lay in enumerate(self.layouts):
            L = d.lev[li]
            if not lay["replicated"]:
                rr = [rk[:4] for rk in lay["ranks"]]
                L.ex_xa, L.ex_xb, L.ex_r = (self._halo_desc(f"{k}{li + 1}", lay["nxn"], rr) for k in ("xa", "xb", "r"))
            elif lay["first_replicated"]:
                L.ex_b = self._gather_desc(f"b{li + 1}", lay["nxn"], lay["ranks"][self.rank][4:6])
        d.err = self._comm_peers[self.rank] + 8 * self.W_ERR

    # -- solve ----------------------------------------------------------------------------------------------------------
    def vcycle(self, k_vals, r, z, dot=None):
        call("fem_mg_vcycle", self.plan._h, C.byref(self.desc), _ptr(k_vals), _ptr(r), _ptr(z), _ptr(dot), _stream())

    def fine_step(self, k_vals, b, x, out, mode=2, step=1, dot=None):
        """One level-0 step of the V-cycle on its own: mode 2 = Chebyshev step ``step`` of the smoother, 1 = residual."""
        c1 = self.desc.c1[step] if mode == 2 else 0.0
        c2 = self.desc.c2[step] if mode == 2 else 0.0
        call("fem_mg_fine_step", self.plan._h, C.byref(self.desc), mode, _ptr(k_vals), _ptr(b), _ptr(x), _ptr(out), c1, c2, _ptr(dot), _stream())

    def fine_step_lattice(self, b, x, out, mode=2, step=1, dot=None):
        """``fine_step`` on the lattice stencil k32s (filled by ``to_f32``) instead of the block-CSR matrix."""
        if self.k32s is None:
            raise ValueError("level 0 of this multigrid does not run on the lattice stencil")
        c1 = self.desc.c1[step] if mode == 2 else 0.0
        c2 = self.desc.c2[step] if mode == 2 else 0.0
        call("fem_mg_fine_step_lattice", self.plan._h, C.byref(self.desc), mode, _ptr(b), _ptr(x), _ptr(out), c1, c2, _ptr(dot), _stream())

    def _exchange_p(self):
        if self.part is not None:
            call("fem_mg_exchange_run", C.byref(self.ex_p), _ptr(self.p), C.c_void_p(self.desc.err), _stream())

    def _update_p(self, it):
        """p = z + beta p on the owned DOFs only: the ghost rows of p belong to the neighbours' pushes."""
        lo, hi = 2 * self.own_nodes[0], 2 * self.own_nodes[1]
        call("fem_mg_pcg_update_p", hi - lo, C.c_void_p(self.z.data_ptr() + 8 * lo), C.c_void_p(self.p.data_ptr() + 8 * lo), _ptr(self.scal), it, _stream())

    def _sum_scal(self, lo, hi):
        """scal[lo:hi] <- sum over the ranks, inside the stream (peer memory, no library call)."""
        if self.part is not None:
            call("fem_peer_allreduce", C.c_void_p(self.scal.data_ptr() + 8 * lo), hi - lo, _ptr(self.comm), self._comm_table, self.W_LINES,
                 self.W_ARSEQ, self.W_ERR, self.rank, self.world, _stream())

    def check_peer_error(self):
        """The sticky time-out word of the in-kernel waits, MAX-reduced so that every rank raises together."""
        if self.part is not None:
            import torch.distributed as dist
            err = self.comm[self.W_ERR:self.W_ERR + 1].clone()
            dist.all_reduce(err, op=dist.ReduceOp.MAX)
            if int(err.item()) != 0:
                raise RuntimeError("multigrid PCG: a peer did not publish within the time-out (tuning key peer_timeout_ms)")

    def _iteration(self, k_vals, it):
        n, s = self.plan.n_dof, self.scal
        self._exchange_p()
        call("fem_pcg_spmv_dot", self.plan._h, _ptr(k_vals), _ptr(self.p), _ptr(self.q), _ptr(self.mask), _ptr(s), it, _stream())
        self._sum_scal(3, 4)
        call("fem_mg_pcg_update_xr", n, _ptr(self.p), _ptr(self.q), _ptr(self.x), _ptr(self.r), _ptr(s), it, _stream())
        slot = 0 if it & 1 else 2
        self.vcycle(k_vals, self.r, self.z, s[slot:slot + 1])
        self._sum_scal(*((1, 3) if it % 2 == 0 else (0, 2)))
        self._update_p(it)

    def launches_per_iteration(self):
        k, L = self.degree, self.n_levels
        return 3 + (2 * k + 3) + (L - 1) * (2 * k + 3) + 1

    def solve(self, k_vals, rhs, rtol=1e-10, maxit=500, check_every=2, iters=None):
        """Returns (x, iterations, relative residual).  ``iters``: run exactly that many iterations (benchmarks)."""
        if self.desc is None:
            self.setup(k_vals)
        P, s, n = self.plan, self.scal, self.plan.n_dof
        self.block_jacobi(k_vals)
        self.to_f32(k_vals)
        call("fem_mg_pcg_init", n, _ptr(rhs), _ptr(self.mask), _ptr(self.r), _ptr(self.x), _ptr(s), _stream())
        self._sum_scal(0, 5)
        self.vcycle(k_vals, self.r, self.z, s[0:1])
        self._sum_scal(0, 1)
        self._update_p(-1)
        n_it = iters if iters is not None else maxit
        it, rel = 0, float("inf")
        h = s.cpu()
        bb = float(h[4])
        if iters is None and (bb == 0.0 or float(h[1]) <= rtol * rtol * bb):
            return self.x, 0, 0.0 if bb == 0.0 else (float(h[1]) / bb) ** 0.5
        graph = None
        if self.use_graph and n_it >= 4:
            if self._graph is None or self._graph_key != k_vals.data_ptr():
                # iterations 0 and 1 run eagerly (they count), then the same pair is captured - capturing does not execute.
                # (No save / restore of the iterates around a warm-up: writing this rank's ghost rows of p back would race
                # with the neighbours' peer stores into them.)
                self._iteration(k_vals, 0)
                self._iteration(k_vals, 1)
                it = 2
                self._capture_pair(k_vals)
            graph = self._graph
        self.launches_last = 0
        # Convergence checks cost a host round trip during which the GPU idles (and a MAX-reduction of the error word across the
        # ranks).  Successive solves of a Newton loop take almost the same number of iterations, so the checks start four
        # iterations before the count of the previous solve on this object; the stopping rule itself is unchanged (the first
        # check that finds rel <= rtol ends the solve - a solve that converges much faster than its predecessor runs a few
        # iterations more than it needed).
        hint = getattr(self, "_hint_iters", {}).get(rtol)              # per tolerance: a looser solve says nothing about a tighter one
        skip_until = 0 if iters is not None else check_schedule(hint, check_every)
        while it < n_it:
            nxt = n_it if iters is not None else next_check(it, n_it, check_every, skip_until)
            while it < nxt:
                if graph is not None and it % 2 == 0 and it + 2 <= nxt:
                    graph.replay()
                    it += 2
                else:
                    self._iteration(k_vals, it)
                    it += 1
            h = s.cpu()
            self.check_peer_error()
            if not torch.isfinite(h[1]):
                raise ArithmeticError("multigrid PCG breakdown: residual is not finite")
            rel = float((h[1] / h[4]).sqrt()) if h[4] > 0 else 0.0
            if iters is None and rel <= rtol:
                break
        self.launches_last = it * self.launches_per_iteration()
        if self.part is not None:
            self.part.halo_exchange(self.x)
        if iters is None and not rel <= rtol:
            from .distributed import PCGNotConverged
            raise PCGNotConverged("multigrid PCG", it, rel, rtol)
        if iters is None:
            self.__dict__.setdefault("_hint_iters", {})[rtol] = it
        return self.x, it, rel

    def _capture_pair(self, k_vals):
        """CUDA graph of an (even, odd) iteration pair: the kernels depend only on the parity of the iteration index, and
        every exchange counter lives on the device, so one graph serves the whole solve (and later solves with the same
        matrix buffer).  Called right after the same two iterations ran eagerly (modules loaded, nothing lazy left)."""
        try:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._iteration(k_vals, 0)
                self._iteration(k_vals, 1)
            self._graph, self._graph_key = g, k_vals.data_ptr()
        except Exception as e:                            # capture unsupported: eager launches
            self.graph_error, self.use_graph, self._graph = repr(e), False, None
