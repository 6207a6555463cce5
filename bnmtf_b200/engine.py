"""Device-side state and sweep driver for the two-factor model (R ~ U V^T).

PyTorch is used for exactly four things here: allocating fp64/int32 device buffers, host<->device copies, the
current CUDA stream, and (row-sharded runs) torch.distributed collectives over NCCL.  Every arithmetic step is a
call into libbnmtf_b200.so through ctypes (bnmtf_b200/_lib.py).

Multi-GPU layout ("dual R / R^T"): rank p owns rows [lo_I, lo_I+cnt_I) of R for the U phase and rows
[lo_J, lo_J+cnt_J) of R^T for the V phase; U and V are replicated.  Rows are conditionally independent inside a
phase, so each rank runs the same kernels on its shard and the only exchanges per sweep are an all-gather of the new
factor rows after each phase and one all-reduce of the metric / ELBO partial sums.
"""
import os
import threading

import numpy as np
import torch

from . import _lib

MODE = {"gibbs": 0, "vb": 1, "icm": 2}
# per-thread switches: DevicePool workers set no_graph (stream capture is process-global: a capture on one thread is
# invalidated by allocations and function-attribute calls made by the fits running on the other threads)
thread_flags = threading.local()
TRACE_COLS = ("tau", "MSE", "R^2", "Rp", "ELBO", "sum_e2", "exp_square_diff", "explogtau")
S_TAU, S_LOGTAU, S_ALPHA_S, S_BETA_S, S_SUM_E2, S_ESD, S_MSE, S_R2, S_RP, S_ELBO = range(10)


_capture_streams = {}


def capture_graph(body):
    """Record the launches body() makes into a CUDA graph (not executed).  torch.cuda.graph() would do the same after a
    device synchronisation, gc.collect() and empty_cache() -- tens of milliseconds, which is longer than a whole toy-size
    run; here only the stream switch capture needs (a side stream per device, ordered after the current one)."""
    dev = torch.cuda.current_device()
    side = _capture_streams.get(dev)
    if side is None:
        side = _capture_streams[dev] = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()
    side.wait_stream(main)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        g.capture_begin()
        try:
            body()
        finally:
            g.capture_end()
    main.wait_stream(side)
    return g


def require_cuda(device=None):
    if not torch.cuda.is_available():
        raise _lib.BnmtfError("no CUDA device visible: bnmtf_b200 has no CPU path")
    _lib.load()
    return torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())


def _ptr(t, row=0):
    """Device address of tensor t (optionally of its row `row`); 0 for None."""
    if t is None:
        return 0
    return t.data_ptr() + (row * t.stride(0) * t.element_size() if row else 0)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def ld_for(n):
    return (int(n) + 63) // 64 * 64


def kp_for(K):
    return 8 * ((K + 1 + 7) // 8)


def gram_len(K):
    nt = kp_for(K) // 8
    return nt * (nt + 1) // 2 * 64


def _pick_nseg(units, ktiles, t_tile, t_fix, sms=148, nmax=32):
    """Number of column segments for a tensor-bound kernel whose grid is `units` x nseg CTAs of one per SM: minimise
    waves x (stages per CTA x t_tile + t_fix) [us] over the segment counts that leave no segment empty."""
    best = None
    for n in range(1, min(ktiles, nmax) + 1):
        tps = -(-ktiles // n)
        if -(-ktiles // tps) != n:
            continue
        cost = -(-(units * n) // sms) * (tps * t_tile + t_fix)
        if best is None or cost < best[0] - 1e-9:
            best = (cost, n)
    return best[1]


class Partition:
    """Contiguous equal-size row shards: rank p owns [lo(p), lo(p)+cnt(p)); the last shards may be short or empty."""

    def __init__(self, n, world=1, rank=0):
        self.n, self.world, self.rank = int(n), int(world), int(rank)
        self.S = -(-self.n // self.world)
        self.n_pad = self.S * self.world

    def lo(self, rank=None):
        return min(self.n, (self.rank if rank is None else rank) * self.S)

    def cnt(self, rank=None):
        return max(0, min(self.S, self.n - self.lo(rank)))


class Comm:
    """The two exchanges of a sharded sweep.  world == 1: no-ops."""

    def __init__(self, world=1, rank=0, group=None):
        self.world, self.rank, self.group = world, rank, group
        self.sync = None           # (sync block, device table of every rank's block, epochs, ...) once setup_sync() ran

    def gather_rows(self, full, part):
        """full: (part.n_pad, ...) tensor whose rows [rank*S, rank*S+S) hold this rank's fresh values -> all ranks'."""
        if self.world == 1:
            return
        import torch.distributed as dist
        S = part.S
        mine = full[self.rank * S:(self.rank + 1) * S].clone()
        dist.all_gather_into_tensor(full[:part.n_pad], mine, group=self.group)

    def allreduce(self, t):
        if self.world == 1:
            return
        if self.sync is not None and t.dtype == torch.float64 and t.numel() <= 32 and t.is_contiguous():
            # <= 32 doubles: our own kernel over the peer-mapped sync blocks (csrc/peer.cu; rank-ordered sum, identical
            # on every rank, capturable in the sweep's CUDA graph)
            _lib.call("bnmtf_peer_sync_f64", _ptr(self.sync[1]), _ptr(self.sync[2]), self.world, self.rank, 2,
                      _ptr(t), t.numel(), _stream())
            return
        import torch.distributed as dist
        dist.all_reduce(t, group=self.group)

    def barrier(self, channel):
        """Cross-GPU barrier on the current stream (after it, every rank sees what every rank wrote before it)."""
        if self.world == 1:
            return
        if self.sync is not None:
            _lib.call("bnmtf_peer_sync_f64", _ptr(self.sync[1]), _ptr(self.sync[2]), self.world, self.rank, int(channel),
                      0, 0, _stream())
            return
        import torch.distributed as dist
        dist.barrier(group=self.group)

    def setup_sync(self, device):
        """One sync block per rank in symmetric memory + a private epoch array (include/bnmtf_b200.h, bnmtf_peer_sync_f64).
        Called by the engine once the fused peer exchange is in use."""
        if self.sync is None and self.peer_enabled(device):
            n = _lib.call("bnmtf_peer_sync_bytes") // 8
            t, hdl, ptrs, keep = self.symmetric((n,), device)
            epoch = torch.zeros(8, dtype=torch.int64, device=device)
            self.sync = (t, ptrs, epoch, keep, hdl)
        return self.sync is not None

    def put_rows(self, full, part, peers_ptrs):
        """This rank's rows of the replicated array `full` -> every other rank's copy (NVLink P2P stores); the caller
        follows up with barrier()."""
        lo, cnt = part.lo(), part.cnt()
        if self.world == 1 or cnt == 0:
            return
        w = full.shape[1] if full.dim() > 1 else 1
        _lib.call("bnmtf_peer_put_f64", _ptr(full, lo), _ptr(peers_ptrs), lo * w, cnt * w, self.world, self.rank, _stream())

    # ---- fused exchange over peer memory (NVLink P2P stores from inside the solver kernel) ------------------------
    def peer_enabled(self, device):
        """True when the updated factor rows are exchanged by the solver kernel itself: world > 1, CUDA + NCCL group,
        BNMTF_PEER != 0.  The NCCL all-gather of gather_rows() stays as the path for everything else (mu / tau on
        demand, gloo on CPU) and as the fallback when symmetric memory cannot be set up on this system."""
        if self.world == 1 or device.type != "cuda" or os.environ.get("BNMTF_PEER", "1") == "0":
            return False
        import torch.distributed as dist
        return dist.is_initialized() and dist.get_backend(self.group) == "nccl"

    def symmetric(self, shape, device):
        """A zeroed fp64 tensor of `shape` allocated in symmetric memory and peer-mapped on every rank of the group
        (torch.distributed._symmetric_memory: allocation, handle exchange and the cross-GPU barrier are torch's; the
        stores into the peers' copies are ours, csrc/solve.cu).  Returns (tensor, handle, device array of the world
        base pointers of this tensor on every rank).  The mapping is verified once by reading a probe value each rank
        writes into its own copy."""
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        group = self.group if self.group is not None else dist.group.WORLD
        t = symm.empty(tuple(shape), dtype=torch.float64, device=device)
        hdl = symm.rendezvous(t, group)
        flat = t.view(-1)
        flat.zero_()
        flat[0] = float(self.rank + 1)
        hdl.barrier(channel=0)
        peers = [t if r == self.rank else hdl.get_remote_tensor(r, tuple(shape), torch.float64) for r in range(self.world)]
        seen = [float(p.view(-1)[0].item()) for p in peers]
        if seen != [float(r + 1) for r in range(self.world)]:
            raise _lib.BnmtfError("symmetric-memory peer mapping check failed: read %s" % seen)
        hdl.barrier(channel=0)
        flat[0] = 0.0
        torch.cuda.synchronize(device)
        hdl.barrier(channel=0)
        ptrs = torch.tensor([p.data_ptr() for p in peers], dtype=torch.int64, device=device)
        return t, hdl, ptrs, peers


class Dataset:
    """This rank's shards of R and of its observation mask on the device, in both orientations (row phase:
    cnt_I x ld(J); column phase: cnt_J x ld(I)), masks as bit words."""

    def __init__(self, I, J, device, world=1, rank=0):
        self.I, self.J, self.device = int(I), int(J), device
        self.ldJ, self.ldI = ld_for(J), ld_for(I)
        self.partI, self.partJ = Partition(I, world, rank), Partition(J, world, rank)
        self.world, self.rank = world, rank
        self.R = self.bits = self.RT = self.bitsT = None
        self.n_obs = None          # global |Omega|
        self.planes = {}           # side -> (digit planes (uint8), row scales) for the tcgen05 R.X kernel, built on demand
        self.wide = {}             # side -> True when some row of that orientation has an outlier (dynamic-range flag)

    def _pack(self, R, M, rows, cols, ld):
        out = torch.zeros((max(rows, 1), ld), dtype=torch.float64, device=self.device)
        bits = torch.zeros((max(rows, 1), ld // 32), dtype=torch.int32, device=self.device)
        if rows > 0:
            Rd = torch.from_numpy(np.ascontiguousarray(R, dtype=np.float64)).to(self.device)
            Md = torch.from_numpy(np.ascontiguousarray(M, dtype=np.float64)).to(self.device)
            _lib.call("bnmtf_pack_dataset_f64", _ptr(Rd), _ptr(Md), rows, cols, ld, _ptr(out), _ptr(bits), _stream())
        return out, bits

    @classmethod
    def from_host(cls, R, M, device=None, world=1, rank=0):
        device = require_cuda(device)
        R = np.asarray(R, dtype=np.float64)
        M = np.asarray(M, dtype=np.float64)
        I, J = R.shape
        ds = cls(I, J, device, world, rank)
        lo, cnt = ds.partI.lo(), ds.partI.cnt()
        ds.R, ds.bits = ds._pack(R[lo:lo + cnt], M[lo:lo + cnt], cnt, J, ds.ldJ)
        if world == 1:
            ds._make_transpose()
        else:
            lo, cnt = ds.partJ.lo(), ds.partJ.cnt()
            ds.RT, ds.bitsT = ds._pack(R[:, lo:lo + cnt].T, M[:, lo:lo + cnt].T, cnt, I, ds.ldI)
        ds.n_obs = float(M.sum())
        return ds

    @classmethod
    def from_device(cls, R_padded, bits, I, J, RT_padded=None, bitsT=None, n_obs=None, world=1, rank=0):
        """Adopt already-resident shards in the library's layout (synthetic benchmark data is generated directly
        on the GPU: a 65536 x 32768 fp64 matrix never exists on the host)."""
        ds = cls(I, J, R_padded.device, world, rank)
        assert R_padded.shape[1] == ds.ldJ and bits.shape[1] == ds.ldJ // 32
        ds.R, ds.bits = R_padded, bits
        if RT_padded is None:
            assert world == 1
            ds._make_transpose()
        else:
            ds.RT, ds.bitsT = RT_padded, bitsT
        ds.n_obs = float(n_obs) if n_obs is not None else None
        return ds

    def _make_transpose(self):
        I, J = self.I, self.J
        self.RT = torch.empty((J, self.ldI), dtype=torch.float64, device=self.device)
        self.bitsT = torch.empty((J, self.ldI // 32), dtype=torch.int32, device=self.device)
        _lib.call("bnmtf_transpose_dataset_f64", _ptr(self.R), _ptr(self.bits), I, J, self.ldJ,
                  _ptr(self.RT), _ptr(self.bitsT), self.ldI, _stream())

    def ensure_planes(self, side):
        """Seven 8-bit digit planes of this rank's rows of R (side 0) / R^T (side 1): the A operand of
        bnmtf_stats_rx_umma_f64.  Built once per dataset (14 GiB per orientation at 65536 x 32768)."""
        if side not in self.planes:
            R, bits = (self.R, self.bits) if side == 0 else (self.RT, self.bitsT)
            rows = (self.partI if side == 0 else self.partJ).cnt()
            ld = self.ldJ if side == 0 else self.ldI
            if rows == 0:
                self.planes[side] = (None, None)
                self.wide[side] = False
                return self.planes[side]
            nbytes = _lib.call("bnmtf_rx_planes_bytes", rows, ld)
            buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
            off = (-buf.data_ptr()) % 1024
            planes = buf[off:off + nbytes]
            rscale = torch.empty(rows, dtype=torch.float64, device=self.device)
            rexp = torch.empty(rows, dtype=torch.int32, device=self.device)
            wide = torch.zeros(1, dtype=torch.int32, device=self.device)
            _lib.call("bnmtf_rx_planes_pack_f64", _ptr(R), _ptr(bits), rows, ld, planes.data_ptr(), _ptr(rscale),
                      _ptr(rexp), _ptr(wide), _stream())
            self.planes[side] = (planes, rscale, buf)
            # outlier rows (typical entry > 2^20 below the largest) keep few bits under one fixed-point scale per row
            self.wide[side] = bool(int(wide.item()))
        return self.planes[side]

    def pack_mask(self, M):
        """Bit-pack this rank's rows of another I x J 0/1 mask (predict(M_pred))."""
        lo, cnt = self.partI.lo(), self.partI.cnt()
        return self._pack(np.zeros((cnt, self.J)), np.asarray(M, dtype=np.float64)[lo:lo + cnt], cnt, self.J, self.ldJ)[1]


class Factor:
    """One factor matrix (n x K, replicated on every rank) with its variational / conditional parameters and its
    padded image.  Arrays have part.n_pad rows so that equal-size shards can be all-gathered in place."""

    def __init__(self, part, K, device, vb, comm=None):
        self.part, self.n, self.K = part, part.n, K
        z = lambda: torch.zeros((part.n_pad, K), dtype=torch.float64, device=device)
        self.peer = None           # (handle, device array of peer base pointers of fac, ... of var) when the solver
        if comm is not None and comm.peer_enabled(device):          # kernel exchanges the rows itself
            try:
                self.fac, hdl, pf, keep_f = comm.symmetric((part.n_pad, K), device)
                self.var = pv = keep_v = None
                if vb:
                    self.var, _, pv, keep_v = comm.symmetric((part.n_pad, K), device)
                self.peer = (hdl, pf, pv, keep_f, keep_v)
            except _lib.BnmtfError:
                raise
            except Exception as exc:                                  # no symmetric memory on this system: NCCL all-gather
                import warnings
                warnings.warn("bnmtf_b200: symmetric memory unavailable (%s: %s); factor rows are exchanged with NCCL "
                              "all-gathers instead of in-kernel peer stores" % (type(exc).__name__, exc))
                self.peer = None
        if self.peer is None:
            self.fac = z()
            self.var = z() if vb else None
        self.lam = z()
        self.lam.fill_(1.0)
        self.mu, self.tauf = z(), z()
        self.n_alloc = ld_for(self.n) + 8
        KP = kp_for(K)
        self.Xp = torch.zeros((self.n_alloc, KP), dtype=torch.float64, device=device)
        self.Vp = torch.zeros((self.n_alloc, KP), dtype=torch.float64, device=device) if vb else None

    def pad(self):
        _lib.call("bnmtf_pad_factor_f64", _ptr(self.fac), _ptr(self.var), self.n, self.K, self.n_alloc,
                  _ptr(self.Xp), _ptr(self.Vp), _stream())


class BNMFEngine:
    """All device work of bnmf_gibbs_optimised / bnmf_vb_optimised / nmf_icm for one (R, M, K)."""

    def __init__(self, dataset, K, mode, alpha, beta, seed=0, comm=None, gram=None):
        self.ds, self.K, self.mode = dataset, int(K), mode
        # per-row Gram statistics: "umma" = tcgen05 fixed-point kernel (csrc/gram_umma.cu), "dmma" = fp64 mma.sync kernel
        self.gram = gram or os.environ.get("BNMTF_GRAM", "umma")
        assert self.gram in ("umma", "dmma")
        # training metrics of a sweep: "stats" = from the column-phase statistics (no third pass over R; the direct
        # pass runs only when the device-side cancellation guard trips), "direct" = always the pass over R
        # masked R.X statistics: "umma" = tcgen05 digit-plane kernel (csrc/rx_umma.cu, K <= 32), "dmma" = fp64 mma.sync
        self.rx = os.environ.get("BNMTF_RX", "umma" if (self.gram == "umma" and self.K <= 32) else "dmma")
        assert self.rx in ("umma", "dmma") and (self.rx == "dmma" or self.K <= 32)
        self.metrics_mode = os.environ.get("BNMTF_METRICS", "stats" if self.gram == "umma" else "direct")
        self.guard = 1e-5
        # 1: replay the sweep as a CUDA graph (0: launch by launch).  Sharded runs are captured too when the exchange runs
        # over peer memory with our own barrier / all-reduce kernels (csrc/peer.cu) -- with NCCL collectives inside the
        # capture (round 1's BNMTF_GRAPH=2) the process group did not shut down cleanly
        g = int(os.environ.get("BNMTF_GRAPH", "1"))
        self.use_graph = g >= 1 and dataset.world == 1          # sharded: decided below, once the exchange path is known
        self._graph = self._graph_key = self._graph_seen = None
        # SMs given to the R.X kernel when both statistics kernels run concurrently (0: one after the other).  The Gram
        # kernel's work grows with K(K+1)/2, the R.X kernel's with K and never below the time to stream the planes:
        # measured best 64 at K = 20 (127.3 / 129.6 / 127.6 sweeps/s at 72 / 64 / 60), 80 at K = 10 (208 vs 197 at 64),
        # 96 at K = 5 (245 vs 228).  Re-measured after the R.X MMAs shrank to N = 640 columns per k-step at K = 20
        # (profiles/r06_split_sweep.txt, short runs): 64 still best at K = 20 (132.5 vs 131.8 / 131.8 / 130.1 at 56 / 72 /
        # 80: with fewer SMs the R.X kernel outlasts the Gram), K = 10, 24 and 32 within 0.3 % of the values tried
        self.split = int(os.environ.get("BNMTF_SPLIT", "64" if self.K > 16 else ("80" if self.K > 8 else "96")))
        self._side = None
        self.m = MODE[mode]
        self.vb = mode == "vb"
        self.alpha, self.beta, self.seed = float(alpha), float(beta), int(seed) & (2 ** 64 - 1)
        self.comm = comm if comm is not None else Comm(dataset.world, dataset.rank)
        dev = dataset.device
        I, J = dataset.I, dataset.J
        self.U = Factor(dataset.partI, K, dev, self.vb, self.comm)
        self.V = Factor(dataset.partJ, K, dev, self.vb, self.comm)
        if dataset.world > 1 and self.U.peer is not None and self.V.peer is not None and self.comm.setup_sync(dev):
            # fused exchange + our own barrier / all-reduce kernels: the sharded sweep contains no NCCL call and no torch
            # collective, so it is captured and replayed exactly like the single-GPU sweep
            self.use_graph = g >= 1
        self.scalars = torch.zeros(16, dtype=torch.float64, device=dev)
        self.iter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.iter_scratch = torch.zeros(1, dtype=torch.int64, device=dev)
        self.trace = None
        self.trace_cap = 0
        self.trace_base = 0         # value of the (never reset) sweep counter when the current trace was allocated
        self.sweeps_done = 0        # host mirror of self.iter; also the Philox stream id, so it only ever grows
        KP, GL = kp_for(K), gram_len(K)
        # local row ranges of the two phases
        self.loc = {0: (dataset.partI.lo(), dataset.partI.cnt()), 1: (dataset.partJ.lo(), dataset.partJ.cnt())}
        # dynamic-range guards of the fixed-point statistics kernels (include/bnmtf_b200.h, bnmtf_range_guard_f64):
        # static -- a dataset with an outlier row keeps the fp64 R.X kernel; dynamic -- a device flag per phase that makes
        # the gated fp64 kernels recompute the statistics (range_trips counts such phases)
        self.range_guard = self.gram == "umma" and os.environ.get("BNMTF_RANGE_GUARD", "1") != "0"
        self.range_flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self.range_trips = torch.zeros(1, dtype=torch.int64, device=dev)
        self.wide_dataset = False
        if self.rx == "umma":
            for side in (0, 1):
                dataset.ensure_planes(side)
            wide = torch.tensor([int(any(dataset.wide.values()))], dtype=torch.int32, device=dev)
            self.comm.allreduce(wide)
            if int(wide.item()) and os.environ.get("BNMTF_RANGE_GUARD", "1") != "0":
                import warnings
                warnings.warn("bnmtf_b200: some row or column of R has outliers more than 2^20 x its typical entry; the 48-bit "
                              "fixed-point statistics kernels would leave those entries fewer than 28 significant bits, "
                              "using the fp64 kernels for this dataset")
                self.rx = self.gram = "dmma"
                self.wide_dataset, self.range_guard = True, False
                self.metrics_mode = os.environ.get("BNMTF_METRICS", "direct")
        # CTAs per launch: aim for >= 6 waves of resident CTAs (148 SMs x 3 resp. 2 CTAs) so that the tail wave
        # costs little; segments are column ranges whose partial results the solver adds up in order
        self.nseg = {}
        for side, ld in ((0, dataset.ldJ), (1, dataset.ldI)):
            rows = max(1, self.loc[side][1])
            rb = (rows + 127) // 128
            if self.rx == "umma":
                # HBM-bound: enough CTAs to keep ~120 SMs streaming, as few segments as possible beyond that (every
                # CTA pays ~10 us of tensor-memory set-up and pipeline fill)
                kt64 = ld // 64
                nrx = max(1, min(kt64, -(-120 // rb)))
                if rb * (kt64 // 160) >= 444:            # plenty of long CTAs: several waves even out the tail
                    nrx = kt64 // 160
                nrx = -(-kt64 // -(-kt64 // nrx))        # no empty segments
            else:
                nrx = max(1, min(ld // 128, -(-2664 // rb)))
            if self.gram == "umma":
                # CTAs = row blocks (rounded up to whole CTA pairs) x column chunks x segments; aim for ~10 waves of one
                # CTA per SM
                tile = 128 if ld >= 256 else 64
                sums = K if (side == 1 and self.metrics_mode == "stats") else 0
                nch = -(-(K * (K + 1) // 2 + (K if self.vb else 0) + sums) // (512 // _lib.call("bnmtf_fixed_point_digits")))
                ktiles = -(-ld // tile)
                ng = _pick_nseg((rb + 1) // 2 * 2 * nch, ktiles, t_tile=0.55 * tile / 128, t_fix=10.0)
                self.umma_tile = getattr(self, "umma_tile", {})
                self.umma_tile[side] = tile
            else:
                gb = (rows + 7) // 8
                ng = max(1, min(-(-(ld // 32) // 32), -(-592 // gb)))
            nm = max(1, min(ld // 128, -(-1776 // rb)))
            self.nseg[side] = (nrx, ng, nm)
        rI, rJ = max(1, self.loc[0][1]), max(1, self.loc[1][1])
        mrx = max(self.nseg[0][0] * rI, self.nseg[1][0] * rJ)
        mg = max(self.nseg[0][1] * rI, self.nseg[1][1] * rJ)
        f64 = lambda *shape: torch.zeros(shape, dtype=torch.float64, device=dev)
        self.RXpart = f64(mrx, KP)
        self.Gpart = f64(mg, GL)
        self.SVpart = f64(mg, KP) if self.vb else None
        self.Gfull = f64(GL + KP)
        if self.rx == "umma":
            self.wsrx_bytes = max(_lib.call("bnmtf_rx_umma_workspace_bytes", self.K, ld) for ld in (dataset.ldJ, dataset.ldI))
            self.wsrx = torch.zeros(self.wsrx_bytes + 1024, dtype=torch.uint8, device=dev)
            self.wsrx_ptr = (self.wsrx.data_ptr() + 1023) // 1024 * 1024
        if self.gram == "umma":
            self.ws_bytes = max(_lib.call("bnmtf_gram_umma_workspace_bytes", self.K, int(self.vb), ld)
                                for ld in (dataset.ldJ, dataset.ldI))
            self.ws = torch.zeros(self.ws_bytes + 1024, dtype=torch.uint8, device=dev)
            self.ws_ptr = (self.ws.data_ptr() + 1023) // 1024 * 1024
        self.gscratch = f64(296 * (GL + KP))          # bnmtf_gram_full_f64: up to 296 partial results
        self.extra = f64(max(rI, rJ)) if self.vb else None
        self.red = f64(24)          # [0:8] metric sums, [8:16] factor ELBO terms, [16] VB extra term
        self.m8, self.el8, self.ex1, self.sums4 = self.red[0:8], self.red[8:16], self.red[16:17], self.red[17:21]
        self.mpart = f64(((rI + 127) // 128) * self.nseg[0][2] * 8)
        self.nb_terms = 64 if max(rI, rJ) * self.K <= (1 << 17) else 296      # CTAs of the ELBO factor terms
        self.elpart = f64(2 * self.nb_terms * 8) if self.vb else None
        self.sterm = None
        self.order_dev = None
        # static sums of the training mask {sum r, sum r^2, |Omega|} over THIS rank's rows: one full-mode pass, p = 0
        self.statics = f64(3)
        if self.loc[0][1] > 0:
            _lib.call("bnmtf_masked_metrics_f64", _ptr(dataset.R), _ptr(dataset.bits), self.loc[0][1], dataset.ldJ,
                      _ptr(self.U.Xp), _ptr(self.V.Xp), self.K, self.nseg[0][2], 0, _ptr(self.mpart), _ptr(self.m8),
                      0, _stream())
            self.statics.copy_(self.m8[4:7])
        self.statics_global = self.statics.clone()
        self.comm.allreduce(self.statics_global)
        self.mstat = f64(max(rI, rJ), 4)
        self.mstat_part = f64(256)
        self.m8d = f64(8)
        self.flag = torch.zeros(1, dtype=torch.int32, device=dev)
        if dataset.n_obs is None:
            tot = self.statics[2:3].clone()
            self.comm.allreduce(tot)
            dataset.n_obs = float(tot.item())
        self.polarity = 0 if dataset.n_obs >= 0.5 * I * J else 1
        self._set_omega(dataset.n_obs)

    # ---- constants depending on |Omega| ---------------------------------------------------------------
    def _set_omega(self, n_obs):
        from scipy.special import gammaln, psi   # host-side scalar constants only
        self.size_Omega = float(n_obs)
        self.alpha_s = self.alpha + self.size_Omega / 2.0
        self.digamma_alpha_s = float(psi(self.alpha_s))
        self.lgamma_alpha = float(gammaln(self.alpha))
        self.lgamma_alpha_s = float(gammaln(self.alpha_s))

    # ---- pieces ---------------------------------------------------------------------------------------
    def _sides(self, side):
        ds = self.ds
        lo, cnt = self.loc[side]
        if side == 0:
            return self.U, self.V, ds.R, ds.bits, cnt, ds.ldJ, lo
        return self.V, self.U, ds.RT, ds.bitsT, cnt, ds.ldI, lo

    def stats(self, side, need_rx=True, sums=False, timers=None):
        """The statistics kernels of one phase (_stats_kernels) followed by the dynamic-range guard of the fixed-point
        kernels and its gated fp64 recomputation (a few microseconds unless the guard trips)."""
        self._stats_kernels(side, need_rx, sums, timers)
        me, other, R, bits, rows, ld, lo = self._sides(side)
        if not self.range_guard or rows == 0:
            return
        nrx, ng, _ = self.nseg[side]
        _lib.call("bnmtf_range_guard_f64", _ptr(self.Gpart), ng, rows, _ptr(self.Gfull), self.polarity, self.K, other.n,
                  self.ws_ptr, _ptr(self.range_flag), _ptr(self.range_trips), _stream())
        _lib.call("bnmtf_stats_gated_f64", _ptr(self.range_flag), _ptr(R), _ptr(bits), rows, ld, _ptr(other.Xp), _ptr(other.Vp),
                  self.K, self.polarity, nrx, ng, _ptr(self.RXpart) if need_rx else 0, _ptr(self.Gpart),
                  _ptr(self.SVpart), _stream())

    def _stats_kernels(self, side, need_rx=True, sums=False, timers=None):
        """Layer-1 passes for one phase: statistics of this rank's rows of R (side 0) / R^T (side 1) w.r.t. the
        other factor.  sums: also the masked column sums of the other factor (for the statistics-based metrics).
        timers: a list that receives (name, start event, end event) for the two kernels as they run HERE, i.e.
        concurrently on their two streams (profile_sweep)."""
        me, other, R, bits, rows, ld, lo = self._sides(side)
        nrx, ng, _ = self.nseg[side]
        other.pad()
        if rows == 0:
            return
        if self.polarity == 0:
            _lib.call("bnmtf_gram_full_f64", _ptr(other.Xp), _ptr(other.Vp), other.n, self.K, ld,
                      _ptr(self.Gfull), _ptr(self.gscratch), _stream())
        if need_rx and self.split > 0 and self.rx == "umma" and self.gram == "umma":
            # SM split: the persistent, HBM-bound R.X kernel takes `split` SMs (high-priority stream, launched first),
            # the tensor-bound Gram kernel the rest; neither could share an SM's tensor memory with the other
            if self._side is None:
                self._side = torch.cuda.Stream(device=self.ds.device, priority=-1)
                self._ev = [torch.cuda.Event(), torch.cuda.Event()]
            main = torch.cuda.current_stream()
            self._ev[0].record(main)
            self._side.wait_event(self._ev[0])
            tev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timers is not None else None
            with torch.cuda.stream(self._side):
                if tev:
                    tev[0].record(self._side)
                self._rx(side, max_ctas=self.split)
                if tev:
                    tev[1].record(self._side)
                self._ev[1].record(self._side)
            if tev:
                tev[2].record(main)
            self._gram(side, sums)
            if tev:
                tev[3].record(main)
                timers.append(("stats_rx_in_sweep", tev[0], tev[1]))
                timers.append(("stats_gram_in_sweep", tev[2], tev[3]))
            main.wait_event(self._ev[1])
        else:
            if need_rx:
                self._rx(side)
            self._gram(side, sums)

    def _rx(self, side, max_ctas=0):
        me, other, R, bits, rows, ld, lo = self._sides(side)
        nrx = self.nseg[side][0]
        if self.rx == "umma":
            planes, rscale = self.ds.ensure_planes(side)[:2]
            _lib.call("bnmtf_stats_rx_umma_f64", planes.data_ptr(), _ptr(rscale), _ptr(R), _ptr(bits), rows, ld, other.n,
                      _ptr(other.Xp), self.K, nrx, max_ctas, _ptr(self.RXpart), self.wsrx_ptr, self.wsrx_bytes, _stream())
        else:
            _lib.call("bnmtf_stats_rx_f64", _ptr(R), _ptr(bits), rows, ld, _ptr(other.Xp), self.K, nrx,
                      _ptr(self.RXpart), _stream())

    def _gram(self, side, sums=False):
        me, other, R, bits, rows, ld, lo = self._sides(side)
        ng = self.nseg[side][1]
        if self.gram == "umma":
            _lib.call("bnmtf_stats_gram_umma_f64", _ptr(bits), rows, ld, other.n, _ptr(other.Xp), _ptr(other.Vp), self.K,
                      self.polarity, ng, self.umma_tile[side], 1 if sums else 0, _ptr(self.Gpart), _ptr(self.SVpart),
                      self.ws_ptr, self.ws_bytes, _stream())
        else:
            _lib.call("bnmtf_stats_gram_f64", _ptr(bits), rows, ld, _ptr(other.Xp), _ptr(other.Vp), self.K,
                      self.polarity, ng, _ptr(self.Gpart), _ptr(self.SVpart), _stream())

    def solve(self, side, order=None, n_order=None, apply=True, minimum_TN=0.0, want_sterm=False, want_extra=False,
              use_iter=True, gather=True, want_mstat=False):
        me, other, R, bits, rows, ld, lo = self._sides(side)
        nrx, ng, _ = self.nseg[side]
        order_ptr = 0
        if order is not None:
            self.order_dev = torch.tensor(list(order), dtype=torch.int32, device=self.ds.device)
            order_ptr, n_order = _ptr(self.order_dev), len(order)
        elif n_order is None:
            n_order = self.K
        if want_sterm and self.sterm is None:
            self.sterm = torch.zeros((max(self.U.part.n_pad, self.V.part.n_pad), self.K), dtype=torch.float64,
                                     device=self.ds.device)
        fused = gather and apply and me.peer is not None     # the kernel stores the finished rows into the peers' copies
        if rows > 0:
            _lib.call("bnmf_row_solve_f64", self.m, rows, self.K, nrx, ng, self.polarity,
                      _ptr(self.RXpart), _ptr(self.Gpart), _ptr(self.SVpart), _ptr(self.Gfull),
                      _ptr(me.fac, lo), _ptr(me.var, lo), _ptr(me.mu, lo), _ptr(me.tauf, lo), _ptr(me.lam, lo),
                      _ptr(self.scalars), order_ptr, n_order, 1 if apply else 0, float(minimum_TN),
                      self.seed, _ptr(self.iter if use_iter else self.iter_scratch), side, lo,
                      _ptr(self.sterm, lo) if want_sterm else 0, _ptr(self.extra) if want_extra else 0,
                      _ptr(self.mstat) if want_mstat else 0,
                      _ptr(me.peer[1]) if fused else 0, _ptr(me.peer[2]) if (fused and self.vb) else 0,
                      self.comm.world if fused else 0, self.comm.rank,
                      _ptr(self.range_flag) if self.range_guard else 0, _stream())
        if fused:
            self.comm.barrier(side)                   # every rank's rows have landed in every copy before anyone reads
        elif gather and self.comm.world > 1:
            if apply:
                self.comm.gather_rows(me.fac, me.part)
                if self.vb:
                    self.comm.gather_rows(me.var, me.part)
            else:
                self.comm.gather_rows(me.mu, me.part), self.comm.gather_rows(me.tauf, me.part)
                if want_sterm:
                    self.comm.gather_rows(self.sterm, me.part)

    def gather_params(self):
        """mu / tau of both factors are only exchanged when the host asks for them (end of run())."""
        if self.comm.world > 1:
            for f in (self.U, self.V):
                self.comm.gather_rows(f.mu, f.part), self.comm.gather_rows(f.tauf, f.part)

    def metrics(self, bits=None):
        """Masked sums over `bits` (default: the training mask) with the current factors -> self.m8 (global)."""
        self.U.pad()
        self.V.pad()
        self._metrics_padded(self.ds.bits if bits is None else bits)
        self.comm.allreduce(self.m8)

    def _metrics_padded(self, bits, gated=False):
        """Local partial sums over this rank's rows of R -> self.m8 (not yet all-reduced).  gated: -> self.m8d, and
        only if the device flag of the statistics-based metrics is raised."""
        ds = self.ds
        lo, rows = self.loc[0]
        if rows == 0:
            (self.m8d if gated else self.m8).zero_()
            return
        statics = _ptr(self.statics) if bits is ds.bits else 0
        _lib.call("bnmtf_masked_metrics_f64", _ptr(ds.R), _ptr(bits), rows, ds.ldJ, _ptr(self.U.Xp, lo), _ptr(self.V.Xp),
                  self.K, self.nseg[0][2], statics, _ptr(self.mpart), _ptr(self.m8d if gated else self.m8),
                  _ptr(self.flag) if gated else 0, _stream())

    def _vb_terms(self):
        """Local partial sums of the factor-side ELBO terms over this rank's rows of U and V -> self.el8."""
        nb = self.nb_terms
        self.elpart.zero_()
        for i, f in enumerate((self.U, self.V)):
            lo, cnt = self.loc[i]
            if cnt > 0:
                _lib.call("bnmtf_vb_factor_terms_f64", _ptr(f.fac, lo), _ptr(f.var, lo), _ptr(f.mu, lo), _ptr(f.tauf, lo),
                          _ptr(f.lam, lo), cnt * f.K, self.elpart[i * nb * 8:].data_ptr(), nb, _stream())
        _lib.call("bnmtf_reduce8_f64", _ptr(self.elpart), 2 * nb, _ptr(self.el8), _stream())

    def _vb_extra(self):
        rows = self.loc[1][1]
        if rows > 0:
            _lib.call("bnmtf_reduce1_f64", _ptr(self.extra), rows, _ptr(self.ex1), _stream())
        else:
            self.ex1.zero_()

    def finish(self, update_tau=True, record=True):
        # the kernel writes trace row number *iter - trace_win[0] (device-side window: the same launch arguments serve
        # every run that reuses the buffer, so a captured sweep stays valid from one run() to the next)
        trace_ptr = _ptr(self.trace) if (record and self.trace is not None) else 0
        _lib.call("bnmf_finish_sweep_f64", self.m, self.alpha, self.beta, self.digamma_alpha_s, self.lgamma_alpha,
                  self.lgamma_alpha_s, (self.ds.I + self.ds.J) * self.K, _ptr(self.m8), _ptr(self.ex1), _ptr(self.el8),
                  _ptr(self.scalars), trace_ptr, _ptr(self.iter if record else self.iter_scratch),
                  0, self.seed, 1 if update_tau else 0, _ptr(self.trace_win) if record else 0, _stream())
        if record:
            self.sweeps_done += 1

    def refresh_scalars(self, update_tau=True):
        """Recompute metrics / exp_square_diff / ELBO (and optionally tau) for the CURRENT state without advancing
        the sweep counter: initialise(), exp_square_diff(), elbo(), quality() of the white-box API."""
        self.red.zero_()
        if self.vb:
            self.stats(1, need_rx=False)
            self.solve(1, n_order=0, apply=False, want_extra=True, use_iter=False, gather=False)
            self._vb_extra()
            self._vb_terms()
        self.U.pad()
        self.V.pad()
        self._metrics_padded(self.ds.bits)
        self.comm.allreduce(self.red)
        self.finish(update_tau=update_tau, record=False)

    # ---- the sweep ------------------------------------------------------------------------------------
    def sweep(self, minimum_TN=0.0):
        """One iteration of run().  The launch sequence of a sweep is static (about 45 launches, every pointer fixed
        while the trace buffer stays the same, the sweep counter lives on the device), so from the second sweep of a
        run on it is replayed as one CUDA graph: the small kernels between the big ones no longer wait for the host."""
        if self.use_graph and not getattr(thread_flags, "no_graph", False):
            key = (self.trace.data_ptr() if self.trace is not None else 0, float(minimum_TN))
            if self._graph is not None and self._graph_key == key:
                self._graph.replay()
                _lib.launch_count[0] += self._graph_kernels       # a replay launches every kernel node of the capture
                self.sweeps_done += 1
                return
            if self._graph_seen == key:                # second sweep with these arguments (in this run() or an earlier one)
                done, count0 = self.sweeps_done, _lib.launch_count[0]
                g = capture_graph(lambda: self._sweep_eager(minimum_TN))          # captured, not executed
                self._graph_kernels = _lib.launch_count[0] - count0
                _lib.launch_count[0] = count0
                self.sweeps_done = done
                self._graph, self._graph_key = g, key
                g.replay()
                _lib.launch_count[0] += self._graph_kernels
                self.sweeps_done += 1
                return
            self._graph_seen = key
        self._sweep_eager(minimum_TN)

    def _sweep_eager(self, minimum_TN=0.0):
        """All U columns, all V columns, tau, metrics (reference run() bodies), launch by launch."""
        stat = self.metrics_mode == "stats"
        self.stats(0)
        self.solve(0, minimum_TN=minimum_TN)
        self.stats(1, sums=stat)
        self.solve(1, minimum_TN=minimum_TN, want_extra=self.vb, want_mstat=stat)
        self.V.pad()                      # U's padded image is current (made for the column phase)
        if stat:
            rows = self.loc[1][1]
            if rows > 0:
                _lib.call("bnmtf_mstat_reduce_f64", _ptr(self.mstat), rows, _ptr(self.mstat_part), _ptr(self.sums4), _stream())
            else:
                self.sums4.zero_()
        else:
            self._metrics_padded(self.ds.bits)
        if self.vb:
            self._vb_extra()
            self._vb_terms()
        self.comm.allreduce(self.red)     # one exchange for metric sums, ELBO terms and the VB extra term
        if stat:
            _lib.call("bnmtf_metrics_from_sums_f64", _ptr(self.sums4), _ptr(self.statics_global), self.guard,
                      _ptr(self.m8), _ptr(self.flag), _stream())
            self._metrics_padded(self.ds.bits, gated=True)     # returns at once unless the guard tripped
            self.comm.allreduce(self.m8d)
            _lib.call("bnmtf_select_metrics_f64", _ptr(self.flag), _ptr(self.m8d), _ptr(self.m8), _stream())
        self.finish(update_tau=True, record=True)

    def profile_sweep(self, reps=3):
        """Per-kernel CUDA-event timings (ms per launch, mean over reps and over the two phases) of the statistics
        passes and the solver, for the roofline block of bench.py.  Runs real sweeps (the state advances; the trace is
        not written)."""
        stat = self.metrics_mode == "stats"
        names = ("stats_rx", "stats_gram", "row_solve", "masked_metrics")
        acc = {n: 0.0 for n in names}
        count = {n: 0 for n in names}

        def timed(name, fn):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            acc[name] += e0.elapsed_time(e1)
            count[name] += 1
        for _ in range(reps):
            for side in (0, 1):
                me, other, R, bits, rows, ld, lo = self._sides(side)
                other.pad()
                if self.polarity == 0:
                    _lib.call("bnmtf_gram_full_f64", _ptr(other.Xp), _ptr(other.Vp), other.n, self.K, ld,
                              _ptr(self.Gfull), _ptr(self.gscratch), _stream())
                timed("stats_rx", lambda: self._rx(side))
                timed("stats_gram", lambda: self._gram(side, sums=stat and side == 1))
                timed("row_solve", lambda: self.solve(side, want_extra=self.vb and side == 1, gather=False,
                                                      want_mstat=stat and side == 1))
                self.solve(side, n_order=0, apply=True, gather=True)   # exchange only (no column is updated)
            self.V.pad()
            if stat:
                rows = self.loc[1][1]
                if rows > 0:
                    _lib.call("bnmtf_mstat_reduce_f64", _ptr(self.mstat), rows, _ptr(self.mstat_part), _ptr(self.sums4), _stream())
                else:
                    self.sums4.zero_()
            else:
                timed("masked_metrics", lambda: self._metrics_padded(self.ds.bits))
            if self.vb:
                self._vb_extra()
                self._vb_terms()
            self.comm.allreduce(self.red)
            if stat:
                _lib.call("bnmtf_metrics_from_sums_f64", _ptr(self.sums4), _ptr(self.statics_global), self.guard,
                          _ptr(self.m8), _ptr(self.flag), _stream())
            self.finish(update_tau=True, record=False)
        out = {n: acc[n] / max(1, count[n]) for n in names}
        # the same two statistics kernels as they run inside a real sweep: side by side on their two streams (SM split)
        if self.split > 0 and self.rx == "umma" and self.gram == "umma":
            timers, spans = [], []
            for _ in range(reps):
                for side in (0, 1):
                    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    p0.record()
                    self.stats(side, sums=stat and side == 1, timers=timers)
                    p1.record()
                    spans.append((p0, p1))
            torch.cuda.synchronize()
            for name in ("stats_rx_in_sweep", "stats_gram_in_sweep"):
                v = [a.elapsed_time(b) for (n, a, b) in timers if n == name]
                out[name] = sum(v) / max(1, len(v))
            out["stats_phase_in_sweep"] = sum(a.elapsed_time(b) for a, b in spans) / max(1, len(spans))
        out["_meta"] = {"gram": self.gram, "rx": self.rx, "metrics_mode": self.metrics_mode, "split": self.split}
        return out

    # ---- small problems: the whole run as ONE kernel (csrc/small.cu) ----------------------------------------
    def small_cluster(self):
        """Cluster size of the single-kernel sweep for this problem, 0 when it does not qualify (large matrix, K > 16,
        sharded run, BNMTF_SMALL=0)."""
        if getattr(self, "_small_c", None) is None:
            ok = self.comm.world == 1 and os.environ.get("BNMTF_SMALL", "1") != "0"
            self._small_c = int(_lib.call("bnmtf_small_cluster_size", self.ds.I, self.ds.J, self.K, int(self.vb))) if ok else 0
            if self._small_c:
                self._small_partial = torch.zeros(16 * 16 + 32, dtype=torch.float64, device=self.ds.device)   # + stage stamps
        return self._small_c

    def sweep_many(self, sweeps, minimum_TN=0.0, samples=None, times=None, sums=None, orders=None):
        """`sweeps` iterations of run() in one launch (small_cluster() must be non-zero).  all_U / all_V: device tensors
        [sweeps, n, K] that receive the Gibbs draw of every sweep; sums = (sum_U, sum_V, burn_in, thinning): running sums of
        the kept draws instead; times: int64 device tensor of sweeps + 1 timestamps."""
        sU, sV, burn_in, thinning = sums if sums is not None else (None, None, 0, 1)
        all_U, all_V = samples if samples is not None else (None, None)
        trace_ptr = _ptr(self.trace) - self.trace_base * 64 if self.trace is not None else 0
        ds, U, V = self.ds, self.U, self.V
        _lib.call("bnmtf_small_sweeps_f64", self.m, _ptr(ds.R), _ptr(ds.bits), _ptr(ds.RT), _ptr(ds.bitsT), ds.I, ds.J, ds.ldJ, ds.ldI,
                  self.K, _ptr(U.fac), _ptr(U.var), _ptr(U.mu), _ptr(U.tauf), _ptr(U.lam), _ptr(V.fac), _ptr(V.var), _ptr(V.mu),
                  _ptr(V.tauf), _ptr(V.lam), _ptr(self.scalars), trace_ptr, _ptr(self.iter), self.trace_base + self.trace_cap,
                  self.alpha, self.beta, self.digamma_alpha_s, self.lgamma_alpha, self.lgamma_alpha_s, float(minimum_TN),
                  self.seed, int(sweeps), _ptr(all_U), _ptr(all_V), _ptr(sU), _ptr(sV), int(burn_in), int(thinning),
                  _ptr(self._small_partial), _ptr(times), _stream())
        self.sweeps_done += int(sweeps)

    def alloc_trace(self, iterations):
        """Trace rows for the next `iterations` sweeps.  The buffer is kept from run to run while it is large enough (only
        the device-side window moves), so the CUDA graph of a sweep survives across run() calls -- run(1) in a loop, the way
        the reference's convergence experiments and bench.py's end-to-end figure drive a model, replays it too."""
        self.trace_cap = int(iterations)
        if self.trace is None or self.trace.shape[0] < max(1, self.trace_cap):
            self.trace = torch.zeros((max(64, self.trace_cap), 8), dtype=torch.float64, device=self.ds.device)
        self.trace_base = self.sweeps_done
        if getattr(self, "trace_win", None) is None:
            self.trace_win = torch.zeros(2, dtype=torch.int64, device=self.ds.device)
        self.trace_win.copy_(torch.tensor([self.trace_base, self.trace_base + self.trace_cap], dtype=torch.int64))


# ==== sparse input: the observed entries only, in CSR form (csrc/sparse.cu) ==========================================
CSR_CHUNK = 1024        # entries per work item of the CSR statistics kernel: longer rows are split, their chunks added in order
CSR_METRIC_CTAS = 1184  # CTAs (partial results) of bnmtf_csr_metrics_f64: 8 per SM


def csr_work_plan(indptr, chunk=CSR_CHUNK):
    """Static work plan of bnmtf_csr_stats_f64 for the row pointers `indptr` (include/bnmtf_b200.h): every row becomes
    ceil(n_i / chunk) items (one for an empty row); the items of a row with more than one get consecutive chunk slots.
    -> dict of numpy arrays item_begin (int64), item_row, item_slot, heavy_row, heavy_first (int32) and n_slots."""
    indptr = np.asarray(indptr, dtype=np.int64)
    rows = indptr.shape[0] - 1
    lens = np.diff(indptr)
    nch = np.maximum(1, -(-lens // chunk))
    item_row = np.repeat(np.arange(rows, dtype=np.int64), nch)
    first = np.cumsum(nch) - nch
    c = np.arange(item_row.shape[0], dtype=np.int64) - np.repeat(first, nch)
    heavy = nch > 1
    item_slot = np.full(item_row.shape[0], -1, dtype=np.int64)
    in_heavy = heavy[item_row]
    item_slot[in_heavy] = np.arange(int(in_heavy.sum()), dtype=np.int64)
    heavy_first = np.concatenate([[0], np.cumsum(nch[heavy])]).astype(np.int32)
    return {"item_begin": indptr[item_row] + c * chunk, "item_row": item_row.astype(np.int32),
            "item_slot": item_slot.astype(np.int32), "heavy_row": np.nonzero(heavy)[0].astype(np.int32),
            "heavy_first": heavy_first, "n_slots": int(heavy_first[-1]), "chunk": int(chunk)}


class DeviceCSR:
    """One CSR orientation on the device: int64 row pointers, int32 column indices, fp64 values, and the static work
    plan of the statistics kernel."""

    def __init__(self, indptr, indices, data, device, plan=True):
        t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(device)
        self.rows = int(len(indptr) - 1)
        self.nnz = int(indptr[-1])
        self.rowptr, self.colidx, self.val = t(indptr, np.int64), t(indices, np.int32), t(data, np.float64)
        if self.nnz == 0:           # (a valid pointer for the kernels, never read)
            self.colidx, self.val = torch.zeros(1, dtype=torch.int32, device=device), torch.zeros(1, dtype=torch.float64, device=device)
        self.plan = None
        if plan:
            p = csr_work_plan(indptr)
            self.chunk, self.n_items, self.n_slots = p["chunk"], int(p["item_row"].shape[0]), p["n_slots"]
            self.n_heavy = int(p["heavy_row"].shape[0])
            self.item_begin, self.item_row, self.item_slot = t(p["item_begin"], np.int64), t(p["item_row"], np.int32), t(p["item_slot"], np.int32)
            self.heavy_row = t(p["heavy_row"], np.int32) if self.n_heavy else None
            self.heavy_first = t(p["heavy_first"], np.int32)
            self.plan = p

    def nbytes(self):
        ts = [self.rowptr, self.colidx, self.val] + ([self.item_begin, self.item_row, self.item_slot, self.heavy_first]
                                                     + ([self.heavy_row] if self.n_heavy else []) if self.plan else [])
        return sum(x.numel() * x.element_size() for x in ts)

    def metrics(self, Ap, Bp, K, partials, out8, run_flag=None):
        """bnmtf_csr_metrics_f64 over these entries -> out8."""
        nparts = max(1, min(CSR_METRIC_CTAS, -(-self.rows // 8)))
        _lib.call("bnmtf_csr_metrics_f64", _ptr(self.rowptr), _ptr(self.colidx), _ptr(self.val), self.rows, _ptr(Ap), _ptr(Bp),
                  int(K), _ptr(partials), nparts, _ptr(out8), _ptr(run_flag), _stream())


class SparseDataset:
    """The training entries of R on the device, in both orientations: CSR of R for the row phase and CSR of R^T (i.e. the
    CSC of R) for the column phase.  No I x J array exists at any point.  `host_R` keeps the canonical host CSR of every
    stored entry of R (training or not), which predict(M_pred) evaluates on.  Single GPU only."""
    world, rank = 1, 0
    bits = None                 # the training entries (the dense engine's `bits` argument: None selects csr[0])

    def __init__(self, host_R, train, device):
        """host_R: canonical scipy.sparse CSR (sorted indices, no duplicates); train: bool per stored entry, or None (all)."""
        self.I, self.J = host_R.shape
        self.device = device
        self.partI, self.partJ = Partition(self.I), Partition(self.J)
        from .data import training_csr
        self.host_R = host_R
        self.host_train = Rt = training_csr(host_R, train)      # host CSR of the training entries (K-means initialisation)
        RtT = Rt.tocsc()            # scipy's counting sort: column-major with sorted row indices, explicit zeros kept
        self.csr = {0: DeviceCSR(Rt.indptr, Rt.indices, Rt.data, device),
                    1: DeviceCSR(RtT.indptr, RtT.indices, RtT.data, device)}
        self.n_obs = float(Rt.indptr[-1])
        # static sums {sum r, sum r^2, |Omega|} of the training entries: the metric kernel with a zero prediction
        zeros = torch.zeros((max(self.I, self.J) + 8) * 8, dtype=torch.float64, device=device)
        part = torch.zeros(CSR_METRIC_CTAS * 8, dtype=torch.float64, device=device)
        out = torch.zeros(8, dtype=torch.float64, device=device)
        self.csr[0].metrics(zeros, zeros, 1, part, out)
        self.statics = out[4:7].clone()

    def nbytes(self):
        return self.csr[0].nbytes() + self.csr[1].nbytes()

    def pack_mask(self, M_pred):
        """The entries of R on the pattern of M_pred (which must lie inside R's stored entries) as a DeviceCSR, the
        entry set bnmtf_csr_metrics_f64 evaluates predict(M_pred) on."""
        from .data import sparse_selection
        sel = sparse_selection(self.host_R, M_pred, "M_pred")
        R = self.host_R
        rows = np.repeat(np.arange(self.I, dtype=np.int64), np.diff(R.indptr))[sel]
        indptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=self.I))]).astype(np.int64)
        return DeviceCSR(indptr, R.indices[sel], R.data[sel], self.device, plan=False)


class SparseBNMFEngine(BNMFEngine):
    """BNMFEngine on a SparseDataset.  The format decision lives here: the statistics of a phase come from one
    bnmtf_csr_stats_f64 call over the phase's CSR (fp64, polarity 1, one segment: no digit planes, no range guard, no
    unmasked totals), the sweep's metrics from the column-phase statistics with bnmtf_csr_metrics_f64 as the gated direct
    pass.  Everything else -- solver calls, factor handling, the end of the sweep, CUDA-graph replay -- is BNMFEngine's."""

    def __init__(self, dataset, K, mode, alpha, beta, seed=0, comm=None):
        if dataset.world != 1:
            raise ValueError("sparse input runs on one GPU")
        self.ds, self.K, self.mode = dataset, int(K), mode
        self.gram = self.rx = "csr"
        self.metrics_mode = "stats"
        self.guard = 1e-5
        self.polarity = 1
        self.range_guard = False
        self.split = 0
        self.use_graph = int(os.environ.get("BNMTF_GRAPH", "1")) >= 1
        self._graph = self._graph_key = self._graph_seen = None
        self._small_c = 0               # never the single-kernel small path
        self.m, self.vb = MODE[mode], mode == "vb"
        self.alpha, self.beta, self.seed = float(alpha), float(beta), int(seed) & (2 ** 64 - 1)
        self.comm = comm if comm is not None else Comm(1, 0)
        dev = dataset.device
        self.U = Factor(dataset.partI, K, dev, self.vb, self.comm)
        self.V = Factor(dataset.partJ, K, dev, self.vb, self.comm)
        self.scalars = torch.zeros(16, dtype=torch.float64, device=dev)
        self.iter = torch.zeros(1, dtype=torch.int64, device=dev)
        self.iter_scratch = torch.zeros(1, dtype=torch.int64, device=dev)
        self.trace, self.trace_cap, self.trace_base, self.sweeps_done = None, 0, 0, 0
        KP, GL = kp_for(K), gram_len(K)
        self.loc = {0: (0, dataset.I), 1: (0, dataset.J)}
        self.nseg = {0: (1, 1, 1), 1: (1, 1, 1)}
        self.range_flag = torch.zeros(1, dtype=torch.int32, device=dev)
        rmax = max(dataset.I, dataset.J)
        smax = max(1, dataset.csr[0].n_slots, dataset.csr[1].n_slots)
        f64 = lambda *shape: torch.zeros(shape, dtype=torch.float64, device=dev)
        self.RXpart, self.Gpart = f64(rmax, KP), f64(rmax, GL)
        self.SVpart = f64(rmax, KP) if self.vb else None
        self.RXc, self.Gc = f64(smax, KP), f64(smax, GL)          # chunk partials of the heavy rows
        self.SVc = f64(smax, KP) if self.vb else None
        self.Gfull = f64(GL + KP)                                    # (read by the solver only at polarity 0)
        self.extra = f64(rmax) if self.vb else None
        self.red = f64(24)
        self.m8, self.el8, self.ex1, self.sums4 = self.red[0:8], self.red[8:16], self.red[16:17], self.red[17:21]
        self.mpart = f64(CSR_METRIC_CTAS * 8)
        self.nb_terms = 64 if rmax * self.K <= (1 << 17) else 296
        self.elpart = f64(2 * self.nb_terms * 8) if self.vb else None
        self.sterm = self.order_dev = None
        self.statics = dataset.statics.clone()
        self.statics_global = self.statics
        self.mstat, self.mstat_part, self.m8d = f64(rmax, 4), f64(256), f64(8)
        self.flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self._set_omega(dataset.n_obs)

    def _sides(self, side):
        lo, cnt = self.loc[side]
        me, other = (self.U, self.V) if side == 0 else (self.V, self.U)
        return me, other, self.ds.csr[side], None, cnt, None, lo

    def stats(self, side, need_rx=True, sums=False, timers=None):
        """RXpart / Gpart / SVpart of one phase from its CSR (the column sums the statistics-based metrics need are in the
        Gram record whatever `sums` says)."""
        me, other, c, _, rows, _, lo = self._sides(side)
        other.pad()
        _lib.call("bnmtf_csr_stats_f64", _ptr(c.rowptr), _ptr(c.colidx), _ptr(c.val), _ptr(c.item_begin), _ptr(c.item_row),
                  _ptr(c.item_slot), c.n_items, c.chunk, _ptr(c.heavy_row), _ptr(c.heavy_first), c.n_heavy, _ptr(other.Xp),
                  _ptr(other.Vp), self.K, _ptr(self.RXpart) if need_rx else 0, _ptr(self.Gpart), _ptr(self.SVpart),
                  _ptr(self.RXc), _ptr(self.Gc), _ptr(self.SVc), _stream())

    def _metrics_padded(self, bits, gated=False):
        """The seven sums over the entry set `bits` (None: the training entries; else a DeviceCSR from pack_mask)."""
        entries = self.ds.csr[0] if bits is None else bits
        entries.metrics(self.U.Xp, self.V.Xp, self.K, self.mpart, self.m8d if gated else self.m8,
                        self.flag if gated else None)

    def small_cluster(self):
        return 0

    def profile_sweep(self, reps=3):
        """CUDA-event timings (ms per call, mean over reps and over the two phases) of the CSR statistics call and the
        solver.  Runs real sweeps (the state advances; the trace is not written)."""
        acc = {"stats_csr_row": 0.0, "stats_csr_col": 0.0, "row_solve": 0.0}
        for _ in range(reps):
            for side in (0, 1):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e[0].record()
                self.stats(side, sums=side == 1)
                e[1].record()
                self.solve(side, want_extra=self.vb and side == 1, want_mstat=side == 1)
                e[2].record()
                e[2].synchronize()
                acc["stats_csr_row" if side == 0 else "stats_csr_col"] += e[0].elapsed_time(e[1]) / reps
                acc["row_solve"] += e[1].elapsed_time(e[2]) / (2 * reps)
            self.V.pad()
            _lib.call("bnmtf_mstat_reduce_f64", _ptr(self.mstat), self.loc[1][1], _ptr(self.mstat_part), _ptr(self.sums4), _stream())
            if self.vb:
                self._vb_extra()
                self._vb_terms()
            _lib.call("bnmtf_metrics_from_sums_f64", _ptr(self.sums4), _ptr(self.statics_global), self.guard,
                      _ptr(self.m8), _ptr(self.flag), _stream())
            self.finish(update_tau=True, record=False)
        acc["stats_csr"] = 0.5 * (acc["stats_csr_row"] + acc["stats_csr_col"])
        acc["_meta"] = {"gram": self.gram, "rx": self.rx, "metrics_mode": self.metrics_mode}
        return acc


def engine_for(dataset, K, mode, alpha, beta, seed=0):
    """The engine that runs on `dataset`: SparseBNMFEngine for a SparseDataset, BNMFEngine otherwise."""
    cls = SparseBNMFEngine if isinstance(dataset, SparseDataset) else BNMFEngine
    return cls(dataset, K, mode, alpha, beta, seed=seed)
