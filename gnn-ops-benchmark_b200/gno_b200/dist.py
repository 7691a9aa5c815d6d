"""Destination-partitioned aggregation across the GPUs of one box (SURVEY §8e).

Destination rows are independent, so they are split into P contiguous ranges, chosen so every
rank gets about the same number of EDGES (power-law graphs concentrate edges on few rows).  Rank r
holds the dst-sorted edge shard of its range, the feature rows of its range, and produces the
output rows of its range.  The one exchange step is an all-gather of the feature shards (NCCL
over NVLink via torch.distributed; gloo in the CPU tests); outputs stay partitioned.

Shards may have different row counts; NCCL all-gather wants equal pieces, so every shard is padded
to `max_rows` and global source ids are remapped once, at plan time, to rows of the padded
[P * max_rows, F] gather buffer.  The partition / remap / exchange logic is device-agnostic torch
(tested with gloo, world_size 2, on CPU); only `aggregate` needs the CUDA library.
"""
import torch
import torch.distributed as dist


def edge_balanced_ranges(row_counts, world):
    """Split rows [0, N) into `world` contiguous ranges with ~equal edge counts.

    row_counts: int64 [N] edges per destination row.  Returns int64 [world + 1] boundaries."""
    n = row_counts.numel()
    csum = torch.cumsum(row_counts.to(torch.int64), 0)
    total = int(csum[-1]) if n else 0
    targets = torch.arange(1, world, dtype=torch.float64, device=row_counts.device) * (total / world)
    cuts = torch.searchsorted(csum.to(torch.float64), targets, right=False) + 1 if n else \
        torch.zeros(world - 1, dtype=torch.int64)
    cuts = cuts.clamp_(max=n).to(torch.int64)
    bounds = torch.cat([torch.zeros(1, dtype=torch.int64, device=cuts.device), cuts,
                        torch.full((1,), n, dtype=torch.int64, device=cuts.device)])
    return torch.cummax(bounds, 0).values  # monotone even for degenerate inputs


def stage_ranges(row_costs, stages, fracs=None):
    """Cut rows [0, n) into `stages` contiguous sub-ranges whose summed cost follows `fracs`
    (default: equal shares).  Returns int64 [stages + 1] boundaries on row_costs' device."""
    n = row_costs.numel()
    if fracs is None:
        fracs = [1.0 / stages] * stages
    if len(fracs) != stages or min(fracs) < 0 or sum(fracs) <= 0:
        raise ValueError("stage_fracs must hold one non-negative share per stage")
    dev = row_costs.device
    csum = torch.cumsum(row_costs.to(torch.float64), 0)
    total = float(csum[-1]) if n else 0.0
    cum = torch.cumsum(torch.tensor(fracs, dtype=torch.float64), 0)[:-1] / sum(fracs)
    cuts = (torch.searchsorted(csum, (cum * total).to(dev), right=False) + 1).clamp_(max=n) if n else \
        torch.zeros(stages - 1, dtype=torch.int64, device=dev)
    bounds = torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), cuts.to(torch.int64),
                        torch.full((1,), n, dtype=torch.int64, device=dev)])
    return torch.cummax(bounds, 0).values


def xorfold_owner(ids, world):
    """Row ownership for power-of-two world sizes: owner = XOR of all log2(world)-bit groups of the
    id, local row = id >> log2(world).  A bijection like cyclic ownership (owner = id % world), but
    balanced on graphs whose id BITS are skewed: every bit of an R-MAT id is 1 with probability
    b + d = 0.24, so under cyclic ownership rank 0 of 2 owns 76 % of the referenced rows."""
    p = world.bit_length() - 1
    if world < 1 or (1 << p) != world:
        raise ValueError("ownership='xorfold' needs a power-of-two world size")
    if p == 0:
        return torch.zeros_like(ids), ids.clone()
    fold = torch.zeros_like(ids)
    t = ids.clone()
    while bool((t != 0).any()) if ids.numel() else False:
        fold ^= t & (world - 1)
        t = t >> p
    return fold, ids >> p


def xorfold_global_ids(owner, world, n_local, device=None):
    """Global ids of the rows `owner` holds under xorfold ownership, in local-row order."""
    p = world.bit_length() - 1
    j = torch.arange(n_local, dtype=torch.int64, device=device)
    if p == 0:
        return j
    fold_hi, _ = xorfold_owner(j << p, world)     # fold of the id with its low bits zeroed
    return (j << p) | (fold_hi ^ owner)


def partition_graph(src, dst, num_nodes, world):
    """Split a global edge list into per-rank shards by destination range.

    Returns (bounds [world+1], [(src_global_r, dst_local_r) for r in range(world)])."""
    counts = torch.bincount(dst, minlength=num_nodes)
    bounds = edge_balanced_ranges(counts, world)
    owner = torch.searchsorted(bounds[1:].contiguous(), dst, right=True)
    shards = []
    for r in range(world):
        m = owner == r
        shards.append((src[m], dst[m] - bounds[r]))
    return bounds, shards


class DistAggregator:
    """One rank's half of the partitioned aggregation.

    bounds      int64 [P+1] destination-row boundaries (same on every rank)
    feature_bounds  int64 [P+1] ownership of the feature rows (default: same as bounds)
    src_global  int64 [E_r]  global source node of each local edge
    dst_local   int64 [E_r]  destination row inside this rank's range
    stages      K > 1 pipelines the exchange (sum / mean): every shard is cut into K row chunks,
                chunk c of all shards is all-gathered while the edges whose sources lie in chunk
                c-1 are being aggregated (accumulating into the output), so NVLink time hides
                behind HBM time instead of adding to it.
    """

    def __init__(self, bounds, src_global, dst_local, rank=None, world=None, group=None, stages=1,
                 feature_bounds=None, exchange="allgather", cyclic_rows=None, stage_fracs=None,
                 row_weight=0, split="dest", ownership="cyclic", push_blocks=148, push_chunk=0,
                 merge_own=False):
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        self.bounds = bounds.to(torch.int64).cpu()
        self.n_out = int(self.bounds[self.rank + 1] - self.bounds[self.rank])
        # Feature rows may be owned in different ranges than the outputs: edge-balanced
        # destination ranges of a skewed graph have very unequal row counts, and padding every
        # feature shard to the largest would inflate the all-gather; equal feature blocks do not.
        self.xbounds = self.bounds if feature_bounds is None else feature_bounds.to(torch.int64).cpu()
        self.dst_local = dst_local
        if cyclic_rows is not None:
            # Cyclic ownership (row i lives on rank i % P as local row i // P): spreads the hub rows
            # of a skewed graph over all owners, so the needed-rows exchange is balanced on the
            # SENDING side too (with contiguous blocks the owner of the low ids serves every rank).
            n_rows = int(cyclic_rows)
            if ownership == "xorfold":
                owner, local = xorfold_owner(src_global, self.world)
                if n_rows % self.world:
                    raise ValueError("ownership='xorfold' needs a row count divisible by the world size")
                self.n_local = self.max_rows = n_rows // self.world
            elif ownership == "cyclic":
                self.n_local = (n_rows - self.rank + self.world - 1) // self.world
                self.max_rows = (n_rows + self.world - 1) // self.world
                owner = src_global % self.world
                local = torch.div(src_global, self.world, rounding_mode="floor")
            else:
                raise ValueError("ownership must be 'cyclic' or 'xorfold'")
        else:
            rows = self.xbounds[1:] - self.xbounds[:-1]
            self.n_local = int(rows[self.rank])
            self.max_rows = int(rows.max())
            # global source id -> (owner rank, row inside the owner's shard)
            b = self.xbounds.to(src_global.device)
            owner = torch.searchsorted(b[1:].contiguous(), src_global, right=True)
            local = src_global - b[owner]
        if exchange in ("needed", "push"):
            # needed-rows exchanges pipeline over DESTINATION sub-ranges (see _setup_needed)
            self.xstages, stages = max(1, int(stages)), 1
            self.stage_fracs, self.row_weight = stage_fracs, int(row_weight)
            # "mixed[D]" (e.g. "mixed16"): the RECEIVER decides — a rank whose rows average at least D edges (default
            # 16) splits by source (its few rows make the accumulate passes cheap and its short
            # own-source stage needs remote rows early), a rank of many low-degree rows takes the
            # hybrid (one extra pass over its output instead of one per stage; its long own-source
            # stage hides the first, large push).  Owners only serve request lists, so ranks may mix;
            # only the number of stages (barriers) is common.
            if split.startswith("mixed"):
                deg = float(split[5:]) if len(split) > 5 else 16.0
                mine = src_global.numel() / max(self.n_out, 1)
                split = "source" if mine >= deg else "hybrid"
                if split == "hybrid":
                    stage_fracs = None      # stage_fracs describes the source ranks' remote groups
                    self.stage_fracs = None
            if split not in ("dest", "source", "hybrid"):
                raise ValueError("split must be 'dest', 'source', 'hybrid' or 'mixed[min_degree]'")
            self.split = split if self.xstages > 1 else "dest"
            # merge_own (source split): the own-source edges and the edges of the first remote group
            # are reduced in ONE launch that gathers from two buffers (x_local and the receive
            # buffer, gno_segment_reduce_two) — one pass over the output and one rounding of a
            # 16-bit sum fewer than reducing them as two accumulating stages, at the price of
            # waiting for the first (small) push before any reduction starts.
            self.merge_own = bool(merge_own) and self.split == "source" and self.xstages > 2
        self.stages = max(1, min(int(stages), max(self.max_rows, 1)))
        # single-stage layout: row of the padded gather buffer [P * max_rows, F]
        self.src_padded = owner * self.max_rows + local if exchange in ("allgather", "allgather_push") else None
        # K-stage layout: chunk c holds rows [c*mc, c*mc + rows_c) of every shard
        self.mc = -(-self.max_rows // self.stages) if self.max_rows else 1
        self.stage_rows = [max(0, min(self.mc, self.max_rows - c * self.mc)) for c in range(self.stages)]
        if self.stages > 1:
            st = torch.div(local, self.mc, rounding_mode="floor")
            self.stage_edges = []
            for c in range(self.stages):
                m = st == c
                ids = owner[m] * self.stage_rows[c] + (local[m] - c * self.mc)
                self.stage_edges.append((ids, dst_local[m]))
        self._plan = None
        self._gidx = None
        self._stage_plans = None
        self._push_stream = None
        self._push_events = None
        self._row_counts = None
        self.push_blocks = int(push_blocks)
        if push_chunk:      # ring slot bytes of the TMA push (process-wide; 0 keeps the library default)
            from ._lib import check, lib
            check(lib.gno_push_set_chunk(int(push_chunk)))
        self.trace = None   # set to [] to collect (label, cuda event) pairs of one staged step
        self.exchange_mode = exchange
        if exchange in ("needed", "push"):
            self._setup_needed(src_global, owner, local)
            if exchange == "push":
                self._setup_push()
        elif exchange == "allgather_push":
            self._ag_bufs = {}
        elif exchange != "allgather":
            raise ValueError("exchange must be 'allgather', 'allgather_push', 'needed' or 'push'")

    # -- needed-rows-only exchange (SURVEY §8f rank 4), pipelined over destination sub-ranges ------
    def _setup_needed(self, src_global, owner, local):
        """Skewed graphs reference only a fraction of the feature rows from each rank (RMAT-26 at
        P=4: 26 %).  Each rank asks every owner for exactly the rows its edges read; per call the
        owners gather those rows and deliver them in the order of the receiver's gather buffer, so
        the gather index of an edge is just the position of its source in that buffer.

        K > 1 stages, split="dest": this rank's destination rows are cut into K contiguous
        sub-ranges (stage s reduces sub-range s); a needed source row belongs to the FIRST stage
        whose edges read it, and the receive buffer is laid out stage-major, owner-minor.  Stage s of
        the exchange then delivers exactly the rows stage s of the reduction is still missing, so
        the reduction of sub-range s can run while the rows of s+1 are in flight — without
        splitting any output row (every row is written once, by one stage; works for every reduce).

        K > 1 stages, split="source" (sum / mean): the needed SOURCE rows are cut into K groups —
        stage 0 = the rows this rank owns itself (nothing to wait for), stages 1..K-1 = the remote
        rows in order of decreasing reference count (stage_fracs = the share of the remote rows in
        each).  Stage s reduces the edges whose source lies in group s, accumulating into the
        output.  On a skewed graph the first remote group is small in bytes but covers most of the
        edges, so almost all of the exchange hides behind the reduction (the destination split
        cannot avoid that every sub-range needs the hub rows first: measured on RMAT-26 at P=2,
        10 % of the edges already read 42 % of the needed rows).  Cost: each stage re-reads and
        re-writes the output rows it touches, and the 16-bit output is rounded once per stage."""
        P, K = self.world, self.xstages
        dev = src_global.device
        key = owner * self.max_rows + local                      # ascending key = grouped by owner
        uniq, inv = torch.unique(key, return_inverse=True)
        uowner = torch.div(uniq, self.max_rows, rounding_mode="floor")
        req = uniq - uowner * self.max_rows                        # row inside the owner's shard
        n_u = int(uniq.numel())
        if K > 1 and self.split == "source":
            fr = self.stage_fracs if self.stage_fracs is not None else [1.0 / (K - 1)] * (K - 1)
            if len(fr) != K - 1 or min(fr) < 0 or sum(fr) <= 0:
                raise ValueError("split='source': stage_fracs holds one share per REMOTE stage (stages - 1)")
            refs = torch.bincount(inv, minlength=n_u)
            remote = torch.nonzero(uowner != self.rank).flatten()
            by_refs = remote[torch.argsort(refs[remote], descending=True, stable=True)]
            cum = torch.cumsum(torch.tensor(fr, dtype=torch.float64), 0) / sum(fr)
            cuts = [0] + [int(round(float(c) * by_refs.numel())) for c in cum]
            cuts[-1] = by_refs.numel()
            first = torch.zeros(n_u, dtype=torch.int64, device=dev)
            for s_ in range(1, K):
                first[by_refs[cuts[s_ - 1]:cuts[s_]]] = s_
            self.sub_bounds = None
            self.stage_of_edge = first[inv]
            self.src_local = local       # stage 0 gathers this rank's own rows straight from x_local
        elif K > 1 and self.split == "hybrid":
            # stage 0 = the edges whose source this rank owns (read from x_local, nothing to wait
            # for); the remote-source edges are cut by DESTINATION sub-range into stages 1..K-1, each
            # accumulating onto stage 0's result: one extra pass over the output in total, instead of
            # one per stage as in the source split, and every sub-range waits only for the remote
            # rows it reads first
            remote_e = owner != self.rank
            counts = torch.bincount(self.dst_local[remote_e], minlength=self.n_out) + self.row_weight
            self.sub_bounds = stage_ranges(counts, K - 1, self.stage_fracs).cpu()
            sb = self.sub_bounds.to(dev)
            dstage = torch.searchsorted(sb[1:].contiguous(), self.dst_local, right=True).clamp_(max=K - 2)
            stage_e = torch.where(remote_e, dstage + 1, torch.zeros_like(dstage))
            first = torch.full((n_u,), K - 1, dtype=torch.int64, device=dev)
            first.scatter_reduce_(0, inv, stage_e, "amin", include_self=True)
            self.stage_of_edge = stage_e
            self.src_local = local
        elif K > 1:
            counts = torch.bincount(self.dst_local, minlength=self.n_out) + self.row_weight
            self.sub_bounds = stage_ranges(counts, K, self.stage_fracs).cpu()
            sb = self.sub_bounds.to(dev)
            stage_e = torch.searchsorted(sb[1:].contiguous(), self.dst_local, right=True).clamp_(max=K - 1)
            first = torch.full((n_u,), K - 1, dtype=torch.int64, device=dev)
            first.scatter_reduce_(0, inv, stage_e, "amin", include_self=True)
            self.stage_of_edge = stage_e
        else:
            self.sub_bounds = torch.tensor([0, self.n_out], dtype=torch.int64)
            first = torch.zeros(n_u, dtype=torch.int64, device=dev)
            self.stage_of_edge = None
        # receive layout: stage-major, owner-minor, ascending row id inside (uniq is sorted)
        order = torch.argsort(first * P + uowner, stable=True)
        pos = torch.empty_like(order)
        pos[order] = torch.arange(n_u, dtype=torch.int64, device=dev)
        self.src_needed = pos[inv]                                 # per-edge row of the receive buffer
        self.n_needed = n_u
        cnt = torch.bincount(first * P + uowner, minlength=K * P).view(K, P)  # rows I receive [stage, owner]
        self.recv_cnt = [[int(v) for v in row] for row in cnt.tolist()]
        flat = cnt.flatten()
        roff = torch.cumsum(flat, 0) - flat                        # where each (stage, owner) block starts
        self.recv_off = [[int(v) for v in row] for row in roff.view(K, P).tolist()]
        self.stage_row0 = [self.recv_off[s][0] for s in range(K)] + [n_u]
        self.recv_splits = [int(v) for v in cnt.sum(0).tolist()]   # per owner, all stages
        # requests travel grouped by owner (stage-minor inside)
        order_o = torch.argsort(uowner * K + first, stable=True)
        req_by_owner = req[order_o].contiguous()
        if P > 1:
            want_cnt = cnt.t().contiguous()                         # [owner, stage]
            serve_cnt = torch.empty_like(want_cnt)                  # [requester, stage]
            dist.all_to_all_single(serve_cnt, want_cnt, group=self.group)
            want_off = roff.view(K, P).t().contiguous()
            put_off = torch.empty_like(want_off)                    # [requester, stage]: where my rows land there
            dist.all_to_all_single(put_off, want_off, group=self.group)
            self.send_splits = [int(v) for v in serve_cnt.sum(1).tolist()]
            serve = torch.empty(sum(self.send_splits), dtype=torch.int64, device=dev)
            dist.all_to_all_single(serve, req_by_owner, self.send_splits, self.recv_splits, group=self.group)
        else:
            serve_cnt, put_off = cnt.t().contiguous(), roff.view(K, P).t().contiguous()
            self.send_splits = list(self.recv_splits)
            serve = req_by_owner
        # serve list: stage-major, requester-minor (it arrived requester-major, stage-minor)
        sc = serve_cnt.flatten()                                     # block sizes in arrival order (q, s)
        blk_q = torch.arange(P, device=dev).repeat_interleave(K)
        blk_s = torch.arange(K, device=dev).repeat(P)
        tag = torch.repeat_interleave(blk_s * P + blk_q, sc)
        self.serve_rows = serve[torch.argsort(tag, stable=True)].contiguous()
        sc_sq = serve_cnt.t().contiguous()                           # [stage, requester]
        self.serve_cnt = [[int(v) for v in row] for row in sc_sq.tolist()]
        self.serve_stage0 = [0]
        for s_ in range(K):
            self.serve_stage0.append(self.serve_stage0[-1] + sum(self.serve_cnt[s_]))
        self.put_off = [[int(v) for v in row] for row in put_off.t().tolist()]  # [stage][requester]

    def _stage_serve(self, s):
        return self.serve_rows[self.serve_stage0[s]:self.serve_stage0[s + 1]]

    def exchange_needed(self, x_local, out=None, gather_rows=None, stage=None, async_op=False):
        """Gather the rows other ranks asked for and deliver them with one all-to-all per stage
        (all stages when stage is None).  gather_rows(x, rows) defaults to the CUDA row-gather
        kernel (gno_gather_rows); the gloo host-logic tests inject their own, the product has no
        CPU path.  Returns the receive buffer (and the list of async works with async_op)."""
        if x_local.size(0) != self.n_local:
            raise ValueError("x_local must hold this rank's rows")
        if gather_rows is None:
            from . import ops
            gather_rows = lambda x, rows: ops.index_select(x, 0, rows)  # noqa: E731
        if out is None:
            out = torch.empty((self.n_needed, x_local.size(1)), dtype=x_local.dtype, device=x_local.device)
        works = []
        for s in (range(self.xstages) if stage is None else [stage]):
            send = gather_rows(x_local, self._stage_serve(s))
            dst = out[self.stage_row0[s]:self.stage_row0[s + 1]]
            if self.world == 1:
                dst.copy_(send)
                continue
            w = dist.all_to_all_single(dst, send, self.recv_cnt[s], self.serve_cnt[s], group=self.group,
                                       async_op=async_op)
            works.append(w)
        return (out, works) if async_op else out

    # -- needed rows pushed over NVLink by the gather kernel itself -----------------------------
    def _setup_push(self):
        """exchange="push": the owners' gather kernel stores each requested row straight into the
        requester's receive buffer through NVLink peer pointers (torch symmetric memory), instead
        of gathering into a send buffer and calling an all-to-all.  _setup_needed already told
        every owner where its rows start inside each requester's buffer (put_off)."""
        n_max = torch.tensor([self.n_needed], dtype=torch.int64, device=self.serve_rows.device)
        if self.world > 1:
            dist.all_reduce(n_max, op=dist.ReduceOp.MAX, group=self.group)
        self._push_rows_max = max(int(n_max.item()), 1)
        self._push_bufs = {}

    def _push_buffer(self, F, dtype, device):
        key = (F, dtype)
        st = self._push_bufs.get(key)
        if st is None:
            import ctypes
            import torch.distributed._symmetric_memory as symm
            t = symm.empty((self._push_rows_max, F), dtype=dtype, device=device)
            hdl = symm.rendezvous(t, self.group if self.group is not None else dist.group.WORLD)
            ptrs = (ctypes.c_void_p * self.world)(*[int(hdl.buffer_ptrs[q]) for q in range(self.world)])
            stages = []
            for s in range(self.xstages):
                seg = [0]
                for c in self.serve_cnt[s]:
                    seg.append(seg[-1] + c)
                stages.append(((ctypes.c_int64 * (self.world + 1))(*seg),
                               (ctypes.c_int64 * self.world)(*self.put_off[s]), seg))
            st = self._push_bufs[key] = (t, hdl, ptrs, stages)
        return st

    def _push_stage(self, x_local, st, s, max_blocks=0):
        """Launch stage s of the exchange on the current stream: one kernel that reads every row a
        peer needs for its stage s once from local HBM and stores it into that peer's buffer.
        max_blocks caps its grid when it runs beside the reduction (0 = fill the chip)."""
        from ._lib import check, lib
        from .plan import _on_device, _ptr, _stream
        t, hdl, ptrs, stages = st
        seg_c, off_c, seg = stages[s]
        rows = self._stage_serve(s)
        F, es = x_local.size(1), x_local.element_size()
        with _on_device(x_local.device):
            check(lib.gno_push_rows(_ptr(x_local), F * es, x_local.stride(0) * es, _ptr(rows),
                                    rows.numel(), self.world, ptrs, seg_c, off_c, F * es,
                                    seg[(self.rank + 1) % self.world], int(max_blocks),
                                    _stream(x_local.device)))

    def exchange_push(self, x_local):
        """All stages back to back on the current stream (no overlap); returns the receive buffer."""
        if x_local.size(0) != self.n_local:
            raise ValueError("x_local must hold this rank's rows")
        x_local = x_local.contiguous()
        st = self._push_buffer(x_local.size(1), x_local.dtype, x_local.device)
        hdl = st[1]
        hdl.barrier(channel=0)  # every peer is done reading its buffer from the previous call
        for s in range(self.xstages):
            self._push_stage(x_local, st, s)
        hdl.barrier(channel=1)  # every row has landed everywhere
        return st[0][:self.n_needed]

    # -- all-gather by peer stores ---------------------------------------------------------------
    def exchange_allgather_push(self, x_local):
        """The all-gather done by this rank's own kernel: every local row is stored into every
        peer's [P * max_rows, F] buffer (torch symmetric memory) with 16-byte NVLink stores —
        706 GB/s per direction measured against 446 GB/s for the NCCL all-gather at P=2."""
        import ctypes
        import torch.distributed._symmetric_memory as symm
        from ._lib import check, lib
        from .plan import _on_device, _ptr, _stream
        if x_local.size(0) != self.n_local:
            raise ValueError("x_local must hold this rank's rows")
        x_local = x_local.contiguous()
        F, es = x_local.size(1), x_local.element_size()
        key = (F, x_local.dtype)
        st = self._ag_bufs.get(key)
        if st is None:
            t = symm.empty((self.world * self.max_rows, F), dtype=x_local.dtype, device=x_local.device)
            hdl = symm.rendezvous(t, self.group if self.group is not None else dist.group.WORLD)
            ptrs = (ctypes.c_void_p * self.world)(*[int(hdl.buffer_ptrs[q]) for q in range(self.world)])
            seg = (ctypes.c_int64 * (self.world + 1))(*[q * self.n_local for q in range(self.world + 1)])
            off = (ctypes.c_int64 * self.world)(*([self.rank * self.max_rows] * self.world))
            st = self._ag_bufs[key] = (t, hdl, ptrs, seg, off)
        t, hdl, ptrs, seg, off = st
        hdl.barrier(channel=0)
        with _on_device(x_local.device):
            check(lib.gno_push_rows(_ptr(x_local), F * es, x_local.stride(0) * es, None,
                                    self.world * self.n_local, self.world, ptrs, seg, off, F * es,
                                    ((self.rank + 1) % self.world) * self.n_local, 0,
                                    _stream(x_local.device)))
        hdl.barrier(channel=1)
        return t

    # -- exchange -------------------------------------------------------------------------------
    def _padded(self, x_local):
        if x_local.size(0) != self.n_local:
            raise ValueError("x_local must hold this rank's rows")
        if self.n_local == self.max_rows:
            return x_local.contiguous()
        piece = torch.empty((self.max_rows, x_local.size(1)), dtype=x_local.dtype, device=x_local.device)
        piece[:self.n_local].copy_(x_local)  # padding rows are never referenced
        return piece

    def exchange(self, x_local, out=None):
        """All-gather the feature shards into the padded [P * max_rows, F] buffer."""
        F = x_local.size(1)
        piece = self._padded(x_local)
        if out is None:
            out = torch.empty((self.world * self.max_rows, F), dtype=x_local.dtype, device=x_local.device)
        if self.world == 1:
            out.copy_(piece)
            return out
        dist.all_gather_into_tensor(out, piece, group=self.group)
        return out

    def exchange_stages(self, x_local, bufs=None):
        """Issue the K chunk all-gathers asynchronously; returns [(buffer, work)] in stage order."""
        F = x_local.size(1)
        piece = self._padded(x_local)
        res = []
        for c in range(self.stages):
            rows = self.stage_rows[c]
            buf = bufs[c] if bufs is not None else torch.empty((self.world * rows, F), dtype=x_local.dtype,
                                                               device=x_local.device)
            chunk = piece[c * self.mc:c * self.mc + rows]
            if self.world == 1 or rows == 0:
                buf.copy_(chunk)
                res.append((buf, None))
            else:
                res.append((buf, dist.all_gather_into_tensor(buf, chunk, group=self.group, async_op=True)))
        return res

    # -- local aggregation (CUDA library) -------------------------------------------------------
    def plan(self):
        if self._plan is None:
            from . import plan as planmod
            self._plan = planmod.build_plan(self.dst_local, self.n_out)
            ids = self.src_needed if self.exchange_mode in ("needed", "push") else self.src_padded
            self._gidx = self._plan.sorted_ids(ids)
        return self._plan, self._gidx

    def stage_plans(self):
        if self._stage_plans is None:
            from . import plan as planmod
            self._stage_plans = []
            for ids, d in self.stage_edges:
                p = planmod.build_plan(d, self.n_out)
                self._stage_plans.append((p, p.sorted_ids(ids)))
        return self._stage_plans

    def xstage_plans(self):
        """needed / push exchange with K stages: one plan per stage
        [(plan, gidx, eid, row_lo, row_hi, accumulate, two_buffers)].  split="dest": the plan of destination
        sub-range [row_lo, row_hi); split="source": a plan over all rows holding the edges whose
        source lies in group s, accumulated onto the earlier stages.  eid maps a sorted edge back
        to its position in this rank's edge list (the arg outputs)."""
        if self._stage_plans is None:
            from . import plan as planmod
            self._stage_plans = []
            for s in range(self.xstages):
                if self.xstages == 1:
                    p, gidx = self.plan()
                    self._stage_plans.append((p, gidx, p.perm, 0, self.n_out, False, False))
                    continue
                if self.merge_own and s == 0:
                    continue            # reduced together with stage 1
                if self.merge_own and s == 1:
                    where = torch.nonzero(self.stage_of_edge <= 1).flatten()
                    p = planmod.build_plan(self.dst_local[where], self.n_out)
                    own_e = self.stage_of_edge[where] == 0
                    ids = torch.where(own_e, self.src_local[where], self.src_needed[where] + self.n_local)
                    self._stage_plans.append((p, p.sorted_ids(ids), p.sorted_ids(where), 0, self.n_out, False, True))
                    continue
                where = torch.nonzero(self.stage_of_edge == s).flatten()
                if self.split == "source" or (self.split == "hybrid" and s == 0):
                    lo, hi, acc = 0, self.n_out, s > 0
                elif self.split == "hybrid":
                    lo, hi, acc = int(self.sub_bounds[s - 1]), int(self.sub_bounds[s]), True
                else:
                    lo, hi, acc = int(self.sub_bounds[s]), int(self.sub_bounds[s + 1]), False
                p = planmod.build_plan(self.dst_local[where] - lo, hi - lo)
                own = self.split in ("source", "hybrid") and s == 0   # rows of x_local, not of the receive buffer
                gidx = p.sorted_ids((self.src_local if own else self.src_needed)[where])
                eid = p.sorted_ids(where)
                self._stage_plans.append((p, gidx, eid, lo, hi, acc, False))
        return self._stage_plans

    def reduce_stages(self, recv, reduce, out, want_arg=False, arg=None, events=None, x_local=None):
        """The local half of a staged step: every stage plan over the receive buffer (waiting for
        events[s] first when given; split="source" reads stage 0 from x_local and waits for
        nothing).  Also what bench.py times as the kernel-only loop."""
        from . import ops
        cur = torch.cuda.current_stream(recv.device)
        own0 = self.split in ("source", "hybrid") and self.xstages > 1
        if own0 and x_local is None:
            raise ValueError("split='source' reduces stage 0 from x_local")
        plans = self.xstage_plans()
        first = self.xstages - len(plans)     # merge_own: the list starts at exchange stage 1
        for k, (p, gidx, eid, lo, hi, acc, dual) in enumerate(plans):
            s = k + first
            if events is not None and not (own0 and s == 0):
                cur.wait_event(events[s])
            self._mark(f"reduce{s} start", cur)
            if hi == lo or (acc and p.E_valid == 0):
                continue
            own_rows = (own0 and s == 0) or dual
            r = ops.segment_reduce(p, x_local if own_rows else recv, reduce, gidx=gidx, eid=eid,
                                   want_arg=want_arg, x2=recv if dual else None,
                                   arg_fill=self.dst_local.numel(), out=out[lo:hi], accumulate=acc)
            if want_arg:
                arg[lo:hi].copy_(r[1])
            self._mark(f"reduce{s} end", cur)

    def _mark(self, label, stream):
        if self.trace is not None:
            e = torch.cuda.Event(enable_timing=True)
            e.record(stream)
            self.trace.append((label, e))

    def _aggregate_staged(self, x_local, reduce, want_arg, x_full, out):
        """K-stage needed-rows exchange overlapped with the reduction (exchange = push | needed).

        Stage s of the exchange delivers the rows stage s of the reduction still misses; the
        reduction of stage s runs as soon as they have landed, while stage s+1 is in flight.
        The exchange runs on a second, high-priority stream so its CTAs take SM slots as
        reduction CTAs retire instead of queueing behind the whole launch."""
        dev = x_local.device
        F = x_local.size(1)
        self.xstage_plans()
        x_local = x_local.contiguous()
        kred = reduce
        if self.split in ("source", "hybrid"):
            if reduce not in ("sum", "mean") or want_arg:
                raise NotImplementedError(f"split='{self.split}' accumulates across stages: sum / mean only "
                                          "(use split='dest' for min / max / mul)")
            kred = "sum"
        if out is None:
            out = torch.empty((self.n_out, F), dtype=x_local.dtype, device=dev)
        arg = torch.empty((self.n_out, F), dtype=torch.int64, device=dev) if want_arg else None
        cur = torch.cuda.current_stream(dev)
        if self._push_stream is None:
            import os
            self._push_stream = torch.cuda.Stream(dev, priority=int(os.environ.get("GNO_PUSH_PRIORITY", "-1")))
            self._push_events = [torch.cuda.Event() for _ in range(self.xstages + 1)]
        ps, ev = self._push_stream, self._push_events
        ev[-1].record(cur)        # x_local is ready and the previous call's reduction has been issued
        ps.wait_event(ev[-1])
        push = self.exchange_mode == "push"
        if push:
            st = self._push_buffer(F, x_local.dtype, dev)
            recv, hdl = st[0][:self.n_needed], st[1]
        else:
            recv = x_full if x_full is not None else torch.empty((self.n_needed, F), dtype=x_local.dtype, device=dev)
        # split="source": stage 0 holds only rows this rank owns; the reduction gathers them straight
        # from x_local, so stage 0 has no exchange at all (and nothing to wait for)
        local0 = self.split in ("source", "hybrid")
        self._mark("step start", cur)
        with torch.cuda.stream(ps):
            if push:
                hdl.barrier(channel=0)      # every peer is done reading its buffer from the previous call
                self._mark("barrier0 done", ps)
            for s in range(self.xstages):
                if local0 and s == 0:
                    continue
                if push:
                    self._push_stage(x_local, st, s, self.push_blocks)
                    self._mark(f"push{s} done", ps)
                    hdl.barrier(channel=1)  # stage s has landed everywhere
                    self._mark(f"barrier after push{s} done", ps)
                else:
                    self.exchange_needed(x_local, recv, stage=s)
                ev[s].record(ps)
        self.reduce_stages(recv, kred, out, want_arg, arg, events=ev, x_local=x_local)
        if reduce == "mean" and self.split in ("source", "hybrid"):
            if self._row_counts is None:
                self._row_counts = torch.bincount(self.dst_local, minlength=self.n_out).clamp_(min=1)
            out.copy_(out.to(torch.float32) / self._row_counts.to(torch.float32).view(-1, 1))
        return (out, arg) if want_arg else out

    def aggregate(self, x_local, reduce="sum", return_arg=False, x_full=None, out=None, stage_bufs=None):
        """out[range_r] = reduce over local edges of x_global[src]; arg = local edge position."""
        from . import ops
        want_arg = return_arg and reduce in ("min", "max")
        if self.exchange_mode in ("needed", "push") and self.xstages > 1:
            return self._aggregate_staged(x_local, reduce, want_arg, x_full, out)
        if self.stages > 1 and reduce in ("sum", "mean") and not return_arg and \
                self.exchange_mode == "allgather":
            plans = self.stage_plans()
            if out is None:
                out = torch.empty((self.n_out, x_local.size(1)), dtype=x_local.dtype, device=x_local.device)
            pending = self.exchange_stages(x_local, stage_bufs)
            for c, ((buf, work), (p, gidx)) in enumerate(zip(pending, plans)):
                if work is not None:
                    work.wait()  # stream-level wait: later chunks keep flowing over NVLink
                ops.segment_reduce(p, buf, "sum", gidx=gidx, out=out, accumulate=c > 0)
            if reduce == "mean":
                plan, _ = self.plan()
                cnt = (plan.rowptr[1:] - plan.rowptr[:-1]).clamp_(min=1).to(torch.float32)
                out.copy_(out.to(torch.float32) / cnt.view(-1, 1))
            return out
        plan, gidx = self.plan()
        if self.exchange_mode == "allgather_push":
            xf = self.exchange_allgather_push(x_local)
        elif self.exchange_mode == "push":
            xf = self.exchange_push(x_local)
        elif self.exchange_mode == "needed":
            xf = self.exchange_needed(x_local, x_full)
        else:
            xf = self.exchange(x_local, x_full)
        return ops.segment_reduce(plan, xf, reduce, gidx=gidx, eid=plan.perm, want_arg=want_arg,
                                  arg_fill=plan.E, out=out)
