"""Driver of hot path 1 (class_statistics): the sequence of local compute steps and -- when the
samples are sharded over the ranks of a process group -- the collectives between them.

Per-class (count, sum x, sum (x - mu)(x - mu)^T) are additive over samples, so every rank
processes its own rows and three all-reduces make the result global (SURVEY.md section 8e):
max label -> n_classes, [class sums | class counts] in ONE buffer -> global means, Gram partials ->
global covariances. The Gram exchange is the only large one. When every rank keeps only its share of
the classes (`shard_output`), it is a reduce-scatter by class FUSED into the Gram kernel and the
epilogue (`class_gram_peer_reduce`): the kernel runs the classes group by group (one group per owner
rank, the rank's own group last) and bumps a device counter when a group's tiles are final; a side
stream waits on the counter with a stream memory operation and the COPY ENGINE pushes the group's
tiles over NVLink into the owner's peer-mapped receive slot while the tensor cores work on the next
group -- no SM, no collective kernel; after one barrier the owner's epilogue sums the slots in rank
order. With replicated output the packed Gram is all-reduced by NCCL behind the kernel (an overlapped
NCCL variant exists, measured not to pay, see DESIGN.md section 8). The local steps are supplied by an
`ops` object: `CudaStatsOps` (the sm_100a kernels through the C ABI) in the product; the CPU test-suite
injects oracle-backed ops to exercise this host logic under the gloo backend.
"""

import ctypes
import os

import torch

from . import _lib


class CudaStatsOps:
    """Local steps of class_statistics on the current CUDA device (kernels K1, K2a, K2, K3).

    `elem` is the element code of the points: 0 for float32 (the float32 entry points), or
    `_lib.ELEM_CODES[torch.bfloat16 / torch.float16]` (the `*_h` entry points, which widen every element
    to float32 as they load it). Sums, means, Grams and statistics are float32 either way."""

    def __init__(self, elem=0):
        self.lib = _lib.load()
        self.elem = elem
        self.gram_events = None  # set to a list to record (start, end) CUDA events around K2

    def _x_fn(self, name):
        """Entry point `name` for this element type, and the leading (X, ldx[, elem]) arguments it takes."""
        if self.elem == 0:
            return getattr(self.lib, name), lambda X: (_lib.ptr(X), X.stride(0))
        return getattr(self.lib, name + "_h"), lambda X: (_lib.ptr(X), X.stride(0), self.elem)

    def _query(self, name, *args):
        """Host-only size query for this element type (the `*_h` queries take the element code last)."""
        if self.elem == 0:
            return getattr(self.lib, name)(*args)
        return getattr(self.lib, name + "_h")(*args, self.elem)

    def label_max(self, y):
        mx = torch.empty(1, dtype=torch.int64, device=y.device)
        _lib.check(
            self.lib.sqfa_label_max(_lib.ptr(y), y.numel(), _lib.ptr(mx), _lib.stream_ptr(y.device)),
            "sqfa_label_max",
        )
        return mx

    _HOST_SLOTS = 32

    def label_max_host(self, y):
        """max(labels) as a Python int: the kernel stores it in mapped pinned host memory and the
        host waits on an event. No device-to-host copy, so the read does not queue behind bulk
        transfers other streams have on the copy engine (`.item()` would)."""
        if getattr(self, "_host_mx", None) is None:
            self._host_mx = torch.empty(self._HOST_SLOTS, dtype=torch.int64).pin_memory()
            self._host_next = 0
        return self.label_max_wait(self.label_max_begin(y))

    def label_max_begin(self, y):
        """Launch the label maximum; `label_max_wait(token)` returns it. Host work done between the two
        (allocating the outputs for the expected number of classes) overlaps the kernel and the wake-up."""
        if getattr(self, "_host_mx", None) is None:
            self._host_mx = torch.empty(self._HOST_SLOTS, dtype=torch.int64).pin_memory()
            self._host_next = 0
        k = self._host_next
        self._host_next = (k + 1) % self._HOST_SLOTS
        slot = self._host_mx[k : k + 1]
        _lib.check(
            self.lib.sqfa_label_max(_lib.ptr(y), y.numel(), _lib.ptr(slot), _lib.stream_ptr(y.device)),
            "sqfa_label_max",
        )
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(y.device))
        return ev, slot

    @staticmethod
    def label_max_wait(token):
        ev, slot = token
        ev.synchronize()
        return int(slot[0])

    def bucket(self, y, C):
        lib, dev, n = self.lib, y.device, y.numel()
        counts = torch.empty(C + 1, dtype=torch.int64, device=dev)
        offsets = torch.empty(C + 2, dtype=torch.int64, device=dev)
        perm = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        ws_bytes = lib.sqfa_bucket_workspace_bytes(n, C)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(
            lib.sqfa_bucket_labels(
                _lib.ptr(y), n, C, _lib.ptr(counts), _lib.ptr(offsets), _lib.ptr(perm), _lib.ptr(ws), ws_bytes,
                _lib.stream_ptr(dev),
            ),
            "sqfa_bucket_labels",
        )
        return perm[:n], offsets, counts

    def class_sums(self, X, perm, offsets, C, out=None):
        lib, dev = self.lib, X.device
        n, D = X.shape
        sums = torch.empty(C, D, dtype=torch.float32, device=dev) if out is None else out
        ws_bytes = lib.sqfa_class_sums_workspace_bytes(n, D, C)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        fn, xa = self._x_fn("sqfa_class_sums")
        _lib.check(
            fn(*xa(X), _lib.ptr(perm), _lib.ptr(offsets), None, n, D, C, _lib.ptr(sums), 0, _lib.ptr(ws), ws_bytes,
               _lib.stream_ptr(dev)),
            "sqfa_class_sums",
        )
        return sums

    def class_sums_shifted(self, X, perm, offsets, shift, C):
        """sum over each class of (x - shift_c) (streaming accumulator)."""
        lib, dev = self.lib, X.device
        n, D = X.shape
        sums = torch.empty(C, D, dtype=torch.float32, device=dev)
        ws_bytes = lib.sqfa_class_sums_workspace_bytes(n, D, C)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
        fn, xa = self._x_fn("sqfa_class_sums")
        _lib.check(
            fn(*xa(X), _lib.ptr(perm), _lib.ptr(offsets), _lib.ptr(shift), n, D, C, _lib.ptr(sums), 0, _lib.ptr(ws),
               ws_bytes, _lib.stream_ptr(dev)),
            "sqfa_class_sums",
        )
        return sums

    def counts_pack(self, counts, out):
        """counts (int64 [C]) -> out (float32 [2 C]) = [count / 2^20 | count mod 2^20], one launch."""
        _lib.check(self.lib.sqfa_counts_pack(_lib.ptr(counts), counts.numel(), _lib.ptr(out),
                                             _lib.stream_ptr(counts.device)), "sqfa_counts_pack")

    def counts_unpack(self, words):
        C = words.numel() // 2
        counts = torch.empty(C, dtype=torch.int64, device=words.device)
        _lib.check(self.lib.sqfa_counts_unpack(_lib.ptr(words), C, _lib.ptr(counts), _lib.stream_ptr(words.device)),
                   "sqfa_counts_unpack")
        return counts

    def class_means(self, sums, counts):
        C, D = sums.shape
        means = torch.empty_like(sums)
        _lib.check(
            self.lib.sqfa_class_means(
                _lib.ptr(sums), _lib.ptr(counts), None, D, C, _lib.ptr(means), _lib.stream_ptr(sums.device)
            ),
            "sqfa_class_means",
        )
        return means

    def pilot_shift(self, X, perm, offsets, C):
        """Centring vectors of the one-pass path: the mean of the first min(n_c, 32) rows of each class."""
        dev = X.device
        shift = torch.empty(C, X.shape[1], dtype=torch.float32, device=dev)
        fn, xa = self._x_fn("sqfa_class_pilot_shift")
        _lib.check(fn(*xa(X), _lib.ptr(perm), _lib.ptr(offsets), X.shape[1], C, _lib.ptr(shift), _lib.stream_ptr(dev)),
                   "sqfa_class_pilot_shift")
        return shift

    def one_pass_splits(self, X, C):
        """Class-sum partials per class of `class_gram_sums` (0: this shape keeps the two passes)."""
        return self._query("sqfa_class_gram_sum_splits", X.shape[0], X.shape[1], C)

    def class_gram_sums(self, X, perm, offsets, shift, C):
        """`class_gram` (centred on `shift`) whose diagonal tiles also write the class sums of x - shift as
        partials [C, nsplit, D]: the one pass over X of single-device class_statistics. Returns (gram, partials)."""
        dev = X.device
        n, D = X.shape
        nsplit = self._query("sqfa_class_gram_sum_splits", n, D, C)
        gram = torch.empty(C, D, D, dtype=torch.float32, device=dev)
        partials = torch.empty(C, nsplit, D, dtype=torch.float32, device=dev)
        ws_bytes = self._query("sqfa_class_gram_workspace_bytes", n, D, C)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        if self.gram_events is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        fn, xa = self._x_fn("sqfa_class_gram_sums")
        _lib.check(
            fn(*xa(X), _lib.ptr(perm), _lib.ptr(offsets), _lib.ptr(shift), n, D, C, _lib.ptr(gram), _lib.ptr(partials),
               _lib.ptr(ws), ws_bytes, _lib.stream_ptr(dev)),
            "sqfa_class_gram_sums",
        )
        if self.gram_events is not None:
            ev[1].record()
            self.gram_events.append(ev)
        return gram, partials

    def means_from_partials(self, partials, counts, shift):
        """(means, sums): sums = the class sums of x - shift (sum of the partials), means = shift + sums / counts."""
        C, nsplit, D = partials.shape
        sums = torch.empty(C, D, dtype=torch.float32, device=partials.device)
        means = torch.empty_like(sums)
        _lib.check(
            self.lib.sqfa_class_means_from_partials(
                _lib.ptr(partials), nsplit, _lib.ptr(counts), _lib.ptr(shift), D, C, _lib.ptr(sums), _lib.ptr(means),
                _lib.stream_ptr(partials.device),
            ),
            "sqfa_class_means_from_partials",
        )
        return means, sums

    supports_packed = True  # class_gram / finalize understand the packed upper-tile layout

    def packed_is_smaller(self, D, C):
        return self.lib.sqfa_gram_packed_floats(D, C) < C * D * D  # padding to 256 can outweigh the triangle

    def class_gram(self, X, perm, offsets, centre, C, packed=False, done=None, n_groups=0, reserve_sms=0,
                   first_class=0):
        """Upper triangle of sum_{i in c} (x_i - centre_c)(x_i - centre_c)^T per class (tcgen05).

        packed=True returns the flat list of 256 x 256 upper tiles (what ranks all-reduce: about
        half the bytes of (C, D, D)); `finalize(..., packed=True)` consumes it. `done` (int32
        [n_groups], zeroed): completion counters per class group, see sqfa_class_gram."""
        lib, dev = self.lib, X.device
        n, D = X.shape
        if packed:
            gram = torch.empty(lib.sqfa_gram_packed_floats(D, C), dtype=torch.float32, device=dev)
        else:
            gram = torch.empty(C, D, D, dtype=torch.float32, device=dev)
        ws_bytes = self._query("sqfa_class_gram_workspace_bytes", n, D, C)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        if self.gram_events is not None:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
        fn, xa = self._x_fn("sqfa_class_gram")
        _lib.check(
            fn(*xa(X), _lib.ptr(perm), _lib.ptr(offsets), _lib.ptr(centre), n, D, C, _lib.ptr(gram), 2 if packed else 0,
               0, _lib.ptr(done), n_groups, first_class, reserve_sms, _lib.ptr(ws), ws_bytes, _lib.stream_ptr(dev)),
            "sqfa_class_gram",
        )
        if self.gram_events is not None:
            ev[1].record()
            self.gram_events.append(ev)
        return gram

    def _collective_group(self, group, max_ctas):
        """Communicator for the overlapped Gram all-reduce: NCCL limited to as many CTAs as SMs are left
        out of the Gram grid (CTAs beyond that could not start before the Gram kernel ends, and the
        collective would finish only then). A dedicated group when `group` spans all ranks (creating a
        group is collective over the default group); otherwise `group` itself."""
        import torch.distributed as dist

        cache = self.__dict__.setdefault("_coll_groups", {})
        key = (id(group), max_ctas)
        if key not in cache:
            pg = group
            # measured (2 x B200, c2): capping NCCL to the reserved SMs makes the collective 2-4x slower than
            # letting its CTAs share the few free SMs, so no cap by default (SQFA_NCCL_CTAS=n to set one)
            ctas = int(os.environ.get("SQFA_NCCL_CTAS", "0"))
            if ctas > 0 and dist.get_world_size(group) == dist.get_world_size() and dist.get_backend(group) == "nccl":
                try:
                    opts = dist.ProcessGroupNCCL.Options()
                    opts.config.max_ctas = ctas
                    opts.config.min_ctas = 1
                    pg = dist.new_group(ranks=list(range(dist.get_world_size())), backend="nccl", pg_options=opts)
                except Exception:  # older torch / NCCL without per-communicator config
                    pg = group
            cache[key] = pg
        return cache[key]

    def class_gram_overlapped(self, X, perm, offsets, centre, C, group):
        """Packed Gram partials of this rank, all-reduced over `group` WHILE the kernel runs: classes are
        split into groups; a side stream waits (stream memory operation) until the kernel has finished a
        group and all-reduces that group's slice. Returns the reduced packed buffer, valid on the
        current stream."""
        import torch.distributed as dist

        lib, dev = self.lib, X.device
        n, D = X.shape
        main = torch.cuda.current_stream(dev)
        if getattr(self, "_side", None) is None or self._side.device != dev:
            self._side = torch.cuda.Stream(device=dev)
        side = self._side
        G = max(1, min(C, int(os.environ.get("SQFA_GRAM_GROUPS", "5"))))
        reserve = int(os.environ.get("SQFA_GRAM_RESERVE_SMS", "8"))
        coll_group = self._collective_group(group, reserve)
        done = torch.zeros(G, dtype=torch.int32, device=dev)
        zeroed = torch.cuda.Event()
        zeroed.record(main)
        trace = getattr(self, "overlap_trace", None)  # diagnostics: list that receives CUDA events
        if trace is not None:
            t0 = torch.cuda.Event(enable_timing=True)
            t0.record(main)
        gram = self.class_gram(X, perm, offsets, centre, C, packed=True, done=done, n_groups=G, reserve_sms=reserve)
        if trace is not None:
            t1 = torch.cuda.Event(enable_timing=True)
            t1.record(main)
            marks = []
        per_class = gram.numel() // C
        side.wait_event(zeroed)  # the counters are zero before the side stream looks at them
        gram.record_stream(side)
        done.record_stream(side)
        lo = 0
        for g in range(G):
            hi = lo
            while hi < C and (hi * G) // C == g:
                hi += 1
            expected = self._query("sqfa_class_gram_group_signals", n, D, C, G, g)
            _lib.check(
                lib.sqfa_stream_wait_geq(ctypes.c_void_p(side.cuda_stream),
                                         ctypes.c_void_p(done.data_ptr() + 4 * g), int(expected)),
                "sqfa_stream_wait_geq",
            )
            with torch.cuda.stream(side):
                dist.all_reduce(gram[lo * per_class : hi * per_class], group=coll_group)
                if trace is not None:
                    ev = torch.cuda.Event(enable_timing=True)
                    ev.record(side)
                    marks.append(ev)
            lo = hi
        if trace is not None:
            trace.append((t0, t1, marks))
        main.wait_stream(side)
        return gram

    # ---- reduce-scatter by class fused into the Gram kernel and the epilogue (peer-mapped memory) ----
    PEER_SETS = 3  # receive-slot sets, used in turn by consecutive calls (callers pipeline steps over streams)

    def peer_acquire(self, D, C, group):
        """Receive slots for the Gram partials of this rank's classes, one per source rank, mapped into
        every peer's address space (torch symmetric memory: CUDA IPC / fabric handles exchanged through
        the group's store). Collective on first use for a (D, C, group). Returns None when peer mapping
        is unavailable (the caller then all-reduces with NCCL). Also makes the current stream wait until
        the epilogue that last read the slot set handed out has finished (with the collective that
        follows on this stream that orders every peer's next push after it)."""
        import torch.distributed as dist

        if os.environ.get("SQFA_PEER_REDUCE", "1") != "1":
            return None
        cache = self.__dict__.setdefault("_peer_states", {})
        dev = torch.device("cuda", torch.cuda.current_device())
        key = (D, C, id(group), dev.index)
        st = cache.get(key)
        if st is None:
            W, r = dist.get_world_size(group), dist.get_rank(group)
            per_class = self.lib.sqfa_gram_packed_floats(D, C) // C
            shares = [class_share(C, q, W) for q in range(W)]
            stride = max(hi - lo for lo, hi in shares) * per_class
            st = {"ok": False}
            try:
                import torch.distributed._symmetric_memory as symm_mem

                buf = symm_mem.empty(self.PEER_SETS * W * stride, dtype=torch.float32, device=dev)
                hdl = symm_mem.rendezvous(buf, group.group_name)
                peers = [hdl.get_buffer(q, (self.PEER_SETS * W * stride,), torch.float32) for q in range(W)]
                st = {"ok": True, "buf": buf, "hdl": hdl, "peers": peers, "W": W, "rank": r, "shares": shares,
                      "per_class": per_class, "stride": stride, "next": 0, "free": [None] * self.PEER_SETS,
                      "side": torch.cuda.Stream(device=dev), "token": torch.zeros(1, device=dev)}
            except Exception as e:  # no peer access between these devices / torch without symmetric memory
                st["why"] = repr(e)
            # all ranks take the same path: one rank without peer mapping sends everyone to NCCL
            ok = torch.tensor([1.0 if st["ok"] else 0.0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            st["ok"] = bool(ok.item() > 0)
            cache[key] = st
        if not st["ok"]:
            return None
        k = st["next"]
        st["next"] = (k + 1) % self.PEER_SETS
        if st["free"][k] is not None:
            torch.cuda.current_stream(dev).wait_event(st["free"][k])
        return {"state": st, "set": k}

    def class_gram_peer_reduce(self, X, perm, offsets, centre, C, group, lease):
        """This rank's packed Gram partials of all classes; every group of classes is pushed to its owner's
        slot [this rank] as soon as the kernel has finished it. Returns the local packed buffer; after the
        call the current stream has passed a barrier behind which all peers' pushes to this rank landed."""
        import torch.distributed as dist

        lib, dev = self.lib, X.device
        n, D = X.shape
        st, k = lease["state"], lease["set"]
        W, r, shares, per_class, stride = st["W"], st["rank"], st["shares"], st["per_class"], st["stride"]
        main, side = torch.cuda.current_stream(dev), st["side"]
        done = torch.zeros(W, dtype=torch.int32, device=dev)
        zeroed = torch.cuda.Event()
        zeroed.record(main)
        own_lo, own_hi = shares[r]
        # class order: the groups of ranks r+1, r+2, ... and this rank's own classes last
        gram = self.class_gram(X, perm, offsets, centre, C, packed=True, done=done, n_groups=W,
                               first_class=own_hi % C)
        side.wait_event(zeroed)
        gram.record_stream(side)
        done.record_stream(side)
        set_base = k * W * stride
        plan = st.setdefault("plans", {}).get(n)
        if plan is None:  # push order and the counter value that says "group g is final", per row count
            plan = [(g, lo, hi, int(self._query("sqfa_class_gram_group_signals", n, D, C, W, g)))
                    for g, lo, hi in peer_push_schedule(r, W, shares)]
            st["plans"][n] = plan
        for g, lo, hi, expected in plan:
            _lib.check(lib.sqfa_stream_wait_geq(ctypes.c_void_p(side.cuda_stream),
                                                ctypes.c_void_p(done.data_ptr() + 4 * g), expected),
                       "sqfa_stream_wait_geq")
            dst = st["peers"][g].data_ptr() + 4 * (set_base + r * stride)
            src = gram.data_ptr() + 4 * lo * per_class
            _lib.check(lib.sqfa_peer_push(ctypes.c_void_p(dst), ctypes.c_void_p(src), 4 * (hi - lo) * per_class,
                                          ctypes.c_void_p(side.cuda_stream)), "sqfa_peer_push")
        main.wait_stream(side)
        # barrier: a rank enters after its pushes completed, and leaves after everyone entered
        dist.all_reduce(st["token"], group=group)
        return gram

    def finalize_peer(self, gram, means, counts, estimator_id, ddof, want_sm, lease):
        """Epilogue over this rank's classes: sum of the W partials (own packed tiles + received slots)."""
        lib, dev = self.lib, gram.device
        st, k = lease["state"], lease["set"]
        W, r, per_class, stride = st["W"], st["rank"], st["per_class"], st["stride"]
        C, D = means.shape
        c0, c1 = st["shares"][r]
        nc = c1 - c0
        cov = torch.empty(nc, D, D, dtype=torch.float32, device=dev)
        sm = torch.empty(nc, D, D, dtype=torch.float32, device=dev) if want_sm else None
        if nc > 0:
            ws_bytes = lib.sqfa_stats_epilogue_workspace_bytes(nc)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            slots = st["buf"].data_ptr() + 4 * k * W * stride
            _lib.check(
                lib.sqfa_stats_epilogue_reduce(
                    ctypes.c_void_p(gram.data_ptr() + 4 * c0 * per_class), ctypes.c_void_p(slots), stride, W, r,
                    _lib.ptr(means[c0:c1]), None, _lib.ptr(counts[c0:c1]), D, nc, estimator_id, ddof, _lib.ptr(cov),
                    _lib.ptr(sm), _lib.ptr(ws), ws_bytes, _lib.stream_ptr(dev),
                ),
                "sqfa_stats_epilogue_reduce",
            )
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        st["free"][k] = ev
        return cov, sm

    def finalize(self, gram, means, counts, estimator_id, ddof, want_sm, packed=False, class_range=None, centred_sums=None):
        """cov (in place over gram unless it is packed; mirrored), optional OAS shrinkage, second moments.
        `class_range` (c0, c1): only those classes (a rank finalising its share of a sharded result).
        `centred_sums`: the class sums of (x - s) when gram was centred on vectors s other than the means."""
        lib, dev = self.lib, gram.device
        C, D = means.shape
        c0, c1 = (0, C) if class_range is None else class_range
        nc = c1 - c0
        if packed:
            per_class = gram.numel() // max(C, 1)
            gram_part = gram[c0 * per_class : c1 * per_class]
            cov = torch.empty(nc, D, D, dtype=torch.float32, device=dev)
        else:
            gram_part = gram[c0:c1]
            cov = gram_part
        sm = torch.empty(nc, D, D, dtype=torch.float32, device=dev) if want_sm else None
        if nc == 0:
            return cov, sm
        means_part, counts_part = means[c0:c1], counts[c0:c1]
        sums_part = None if centred_sums is None else centred_sums[c0:c1]
        ws_bytes = lib.sqfa_stats_epilogue_workspace_bytes(nc)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(
            lib.sqfa_stats_epilogue(
                _lib.ptr(gram_part), _lib.ptr(means_part), _lib.ptr(sums_part), _lib.ptr(counts_part), D, nc,
                estimator_id | (16 if packed else 0) | (32 if centred_sums is not None else 0), ddof, _lib.ptr(cov), _lib.ptr(sm), _lib.ptr(ws), ws_bytes,
                _lib.stream_ptr(dev),
            ),
            "sqfa_stats_epilogue",
        )
        return cov, sm

    def fused_prepare(self, X, C, want_sm):
        """Outputs and workspace of `fused` for C classes (allocated while the label maximum is in flight)."""
        lib, dev = self.lib, X.device
        n, D = X.shape
        means = torch.empty(C, D, dtype=torch.float32, device=dev)
        cov = torch.empty(C, D, D, dtype=torch.float32, device=dev)
        sm = torch.empty(C, D, D, dtype=torch.float32, device=dev) if want_sm else None
        meta = torch.empty(2 * C + 4, dtype=torch.int64, device=dev)  # counts [C+1] | offsets [C+2]
        perm = torch.empty(n, dtype=torch.int32, device=dev)
        ws_bytes = self._query("sqfa_class_statistics_workspace_bytes", n, D, C)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        return C, want_sm, means, cov, sm, meta, perm, ws, ws_bytes

    def fused(self, X, y, C, estimator_id, ddof, want_sm, prepared=None):
        """All local steps from ONE C call (sqfa_class_statistics): no host work between kernels."""
        lib, dev = self.lib, X.device
        n, D = X.shape
        if prepared is None or prepared[0] != C or prepared[1] != want_sm:
            prepared = self.fused_prepare(X, C, want_sm)
        _, _, means, cov, sm, meta, perm, ws, ws_bytes = prepared
        counts, offsets = meta[: C + 1], meta[C + 1 : 2 * C + 3]
        fn, xa = self._x_fn("sqfa_class_statistics")
        _lib.check(
            fn(*xa(X), _lib.ptr(y), n, D, C, estimator_id, ddof, _lib.ptr(means), _lib.ptr(cov), _lib.ptr(sm),
               _lib.ptr(counts), _lib.ptr(offsets), _lib.ptr(perm), _lib.ptr(ws), ws_bytes, _lib.stream_ptr(dev)),
            "sqfa_class_statistics",
        )
        return means, cov, sm, (perm, offsets, counts)


class CudaStatsOps64(CudaStatsOps):
    """float64 local steps (SURVEY.md 8(f) row 3): DFMA kernels of stats64.cu. Bucketing and the label
    maximum are dtype-independent and inherited; there is no packed Gram and no one-call fused path."""

    supports_packed = False
    class_gram_sums = None  # float64 keeps its two passes
    fused = None
    fused_prepare = None
    counts_pack = None
    class_gram_overlapped = None
    peer_acquire = None

    def class_sums(self, X, perm, offsets, C, out=None):
        n, D = X.shape
        sums = torch.empty(C, D, dtype=torch.float64, device=X.device) if out is None else out
        _lib.check(
            self.lib.sqfa_class_sums_f64(_lib.ptr(X), X.stride(0), _lib.ptr(perm), _lib.ptr(offsets), None, n, D, C,
                                         _lib.ptr(sums), 0, _lib.stream_ptr(X.device)),
            "sqfa_class_sums_f64",
        )
        return sums

    def class_means(self, sums, counts):
        C, D = sums.shape
        means = torch.empty_like(sums)
        _lib.check(
            self.lib.sqfa_class_means_f64(_lib.ptr(sums), _lib.ptr(counts), None, D, C, _lib.ptr(means),
                                          _lib.stream_ptr(sums.device)),
            "sqfa_class_means_f64",
        )
        return means

    def class_gram(self, X, perm, offsets, centre, C, packed=False, **_unused):
        n, D = X.shape
        gram = torch.empty(C, D, D, dtype=torch.float64, device=X.device)
        _lib.check(
            self.lib.sqfa_class_gram_f64(_lib.ptr(X), X.stride(0), _lib.ptr(perm), _lib.ptr(offsets), _lib.ptr(centre),
                                         n, D, C, _lib.ptr(gram), 0, _lib.stream_ptr(X.device)),
            "sqfa_class_gram_f64",
        )
        return gram

    def finalize(self, gram, means, counts, estimator_id, ddof, want_sm, packed=False, class_range=None):
        C, D = means.shape
        c0, c1 = (0, C) if class_range is None else class_range
        nc = c1 - c0
        dev = gram.device
        cov = torch.empty(nc, D, D, dtype=torch.float64, device=dev)
        sm = torch.empty(nc, D, D, dtype=torch.float64, device=dev) if want_sm else None
        if nc > 0:
            _lib.check(
                self.lib.sqfa_stats_epilogue_f64(_lib.ptr(gram[c0:c1]), _lib.ptr(means[c0:c1]), None,
                                                 _lib.ptr(counts[c0:c1]), D, nc, estimator_id, ddof, _lib.ptr(cov),
                                                 _lib.ptr(sm), _lib.stream_ptr(dev)),
                "sqfa_stats_epilogue_f64",
            )
        return cov, sm


def _all_reduce(t, group, op=None):
    import torch.distributed as dist

    dist.all_reduce(t, op=op if op is not None else dist.ReduceOp.SUM, group=group)


_COUNT_BASE = 1 << 20  # class counts travel as two float32 (hi, lo) next to the class sums: exact below 2^44


def class_share(n_classes, rank, world):
    """Contiguous range of classes whose statistics `rank` finalises when the output is sharded: the
    classes c with c * world // n_classes == rank (the grouping of the Gram kernel's completion counters)."""
    return -((-n_classes * rank) // world), -((-n_classes * (rank + 1)) // world)


def peer_push_schedule(rank, world, shares):
    """Order in which `rank` pushes class groups to their owners in the fused reduce-scatter: the groups of
    ranks rank+1, rank+2, ... (the order the Gram kernel finishes them in, its own group runs last and is
    not pushed). At every step the ranks address pairwise different peers."""
    out = []
    for step in range(1, world):
        g = (rank + step) % world
        lo, hi = shares[g]
        if hi > lo:
            out.append((g, lo, hi))
    return out


def run_class_statistics(ops, X, y, estimator_id, group=None, n_classes=None, ddof=1, centre=None, want_sm=True,
                         shard_output=False):
    """means, covariances, second moments of the labeled rows; with `group`, of the union of the
    rows held by all ranks (every rank returns the full global result, or -- `shard_output` -- the
    means of all classes and the covariances / second moments of its `class_share`).

    On one device without `centre`, ONE pass over the rows: the Gram is centred on a pilot shift (the mean
    of each class's first 32 rows) and writes the class sums of x - shift on the way; mean = shift + sums / n
    and the epilogue takes n d d^T (d = mean - shift) off the Gram. That is what the single call
    `sqfa_class_statistics` runs, step by step. Otherwise two passes over the local rows, like the
    reference (mean first, then the Gram of the centred rows, statistics.py:118-120): a process group
    all-reduces the sums before the Gram so that every rank centres on the same means. `centre` (C, D)
    overrides the centring vectors.
    """
    prepared = None
    if n_classes is None:
        # the one host read the reference also does (statistics.py:29)
        if group is None and getattr(ops, "label_max_host", None) is not None:
            token = ops.label_max_begin(y)
            guess = getattr(ops, "_last_n_classes", None)
            speculative = None
            fusable = (guess and centre is None and y.numel() > 0 and getattr(ops, "fused_prepare", None) is not None
                       and getattr(ops, "fused", None) is not None and getattr(ops, "gram_events", None) is None)
            if fusable and getattr(ops, "_n_classes_streak", 0) < 1:
                # the class count has not repeated yet: only allocate for it while the kernel runs
                prepared = ops.fused_prepare(X, guess, want_sm)
            elif fusable:
                # Do not idle while the label maximum travels to the host: run the whole call for as many
                # classes as the last call had, enqueued right behind the label_max kernel, and check afterwards.
                # A different class count (first call on new data) discards it and runs again below -- any
                # guess is safe to execute: labels beyond it fall into the "dropped" bucket, classes without
                # rows are empty.
                prepared = ops.fused_prepare(X, guess, want_sm)
                speculative = ops.fused(X, y, guess, estimator_id, ddof, want_sm, prepared)
            n_classes = ops.label_max_wait(token) + 1
            ops._n_classes_streak = getattr(ops, "_n_classes_streak", 0) + 1 if n_classes == guess else 0
            ops._last_n_classes = n_classes
            if speculative is not None:
                if n_classes == guess:
                    return speculative
                prepared = None
        else:
            mx = ops.label_max(y)
            if group is not None:
                import torch.distributed as dist

                _all_reduce(mx, group, dist.ReduceOp.MAX)
            if getattr(ops, "label_max_host", None) is not None:
                n_classes = ops.label_max_host(mx) + 1  # max of one element: publishes it to the host
            else:
                n_classes = int(mx.item()) + 1
    C = n_classes
    if (
        group is None and centre is None and C > 0 and y.numel() > 0
        and getattr(ops, "fused", None) is not None and getattr(ops, "gram_events", None) is None
    ):
        return ops.fused(X, y, C, estimator_id, ddof, want_sm, prepared)
    perm, offsets, counts = ops.bucket(y, C)
    D = X.shape[1]
    if (group is None and centre is None and getattr(ops, "class_gram_sums", None) is not None
            and ops.one_pass_splits(X, C) > 0):
        class_counts = counts[:C].clone()
        shift = ops.pilot_shift(X, perm, offsets, C)
        gram, partials = ops.class_gram_sums(X, perm, offsets, shift, C)
        means, sums = ops.means_from_partials(partials, class_counts, shift)
        cov, sm = ops.finalize(gram, means, class_counts, estimator_id, ddof, want_sm, centred_sums=sums)
        return means, cov, sm, (perm, offsets, counts)
    lease = None
    if (group is not None and shard_output and centre is None and getattr(ops, "peer_acquire", None) is not None
            and getattr(ops, "supports_packed", False) and ops.packed_is_smaller(D, C)
            and getattr(ops, "gram_events", None) is None):
        lease = ops.peer_acquire(D, C, group)  # before the collective below (see peer_acquire)
    if group is not None:
        # ONE small collective: [class sums | counts / 2^20 | counts mod 2^20] in the dtype of the sums
        # (float64 for float64 points, float32 otherwise: bf16 / fp16 points have float32 sums)
        sums_dtype = torch.float64 if X.dtype == torch.float64 else torch.float32
        small = torch.empty(C * D + 2 * C, dtype=sums_dtype, device=X.device)
        sums = small[: C * D].view(C, D)
        local_sums = ops.class_sums(X, perm, offsets, C, out=sums)
        if local_sums is not sums:  # ops without an `out` argument
            sums.copy_(local_sums)
        local = counts[:C]
        native_words = small.dtype == torch.float32 and getattr(ops, "counts_pack", None) is not None
        if native_words:  # one launch each way instead of a dozen element-wise torch kernels
            ops.counts_pack(local, small[C * D :])
        else:
            small[C * D : C * D + C] = torch.div(local, _COUNT_BASE, rounding_mode="floor").to(sums_dtype)
            small[C * D + C :] = torch.remainder(local, _COUNT_BASE).to(sums_dtype)
        _all_reduce(small, group)
        if native_words:
            class_counts = ops.counts_unpack(small[C * D :])
        else:
            class_counts = (small[C * D : C * D + C].round().to(torch.int64) * _COUNT_BASE
                            + small[C * D + C :].round().to(torch.int64))
    else:
        sums = ops.class_sums(X, perm, offsets, C)
        class_counts = counts[:C].clone()
    means = ops.class_means(sums, class_counts)
    shift = means if centre is None else centre
    class_range = None
    if group is not None and shard_output:
        import torch.distributed as dist

        class_range = class_share(C, dist.get_rank(group), dist.get_world_size(group))
    extra = {} if class_range is None else {"class_range": class_range}
    packed_ok = group is not None and getattr(ops, "supports_packed", False) and ops.packed_is_smaller(D, C)
    overlap = getattr(ops, "class_gram_overlapped", None) is not None and getattr(ops, "gram_events", None) is None
    # Opt-in (SQFA_GRAM_OVERLAP=1). Measured on 2 x B200 at c2 (tools/sweep_overlap.sh): NCCL's kernels only
    # start once >= 8 SMs are free, leaving 8 SMs out of the Gram grid costs the Gram a whole extra round of
    # tiles (+0.19 ms of 2.0), and the all-reduce progresses at ~45 GB/s on those few SMs -- the step comes
    # out within +-0.06 ms of the serialised version (2.82 vs 2.90 and 2.98 vs 2.92 ms on two boxes).
    if lease is not None:
        # reduce-scatter by class fused into the Gram kernel (copy-engine pushes) and the epilogue
        gram = ops.class_gram_peer_reduce(X, perm, offsets, shift, C, group, lease)
        cov, sm = ops.finalize_peer(gram, means, class_counts, estimator_id, ddof, want_sm, lease)
    elif packed_ok and overlap and os.environ.get("SQFA_GRAM_OVERLAP", "0") == "1":
        # the one large collective, hidden behind the kernel that produces its input
        gram = ops.class_gram_overlapped(X, perm, offsets, shift, C, group)
        cov, sm = ops.finalize(gram, means, class_counts, estimator_id, ddof, want_sm, packed=True, **extra)
    elif packed_ok:
        gram = ops.class_gram(X, perm, offsets, shift, C, packed=True)
        _all_reduce(gram, group)
        cov, sm = ops.finalize(gram, means, class_counts, estimator_id, ddof, want_sm, packed=True, **extra)
    else:
        gram = ops.class_gram(X, perm, offsets, shift, C)
        if group is not None:
            _all_reduce(gram, group)
        cov, sm = ops.finalize(gram, means, class_counts, estimator_id, ddof, want_sm, **extra)
    return means, cov, sm, (perm, offsets, counts)


def pair_range(n_pairs, rank, world):
    """Contiguous slice [begin, end) of the linearised class-pair list owned by `rank`."""
    return (n_pairs * rank) // world, (n_pairs * (rank + 1)) // world
