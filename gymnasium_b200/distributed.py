"""Sharding a vector env across the GPUs of one box (one process per GPU, ``torch.distributed``).

Sub-envs are independent (no cross-env term anywhere on the path), so the global index range is cut into contiguous
shards and each rank steps its own shard with no exchange.  Seeds use the GLOBAL env index (``seed + env_offset + i``) so
results do not depend on the number of ranks.  Two ways to one batch of step outputs:

* :class:`BatchGather` -- on the device, one NCCL gather / all-gather per tensor (NVLink; gloo on CPU in the tests);
* :class:`HostBatch` + :class:`HostBatchPipeline` -- on the host, what ``AsyncVectorEnv`` hands out: every rank maps ONE
  shared page-locked buffer and lands its rows there over its own PCIe link, `depth` steps in flight (a landing kernel
  stores the rows and publishes a per-rank sequence word; the consumer releases slots through an acknowledgement word).
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist


def shard_bounds(total: int, world_size: int, rank: int) -> tuple[int, int]:
    """(start, count) of rank's contiguous shard; the first ``total % world_size`` ranks get one extra env."""
    if not 0 <= rank < world_size:
        raise ValueError(f"rank {rank} outside world of {world_size}")
    base, extra = divmod(int(total), int(world_size))
    start = rank * base + min(rank, extra)
    return start, base + (1 if rank < extra else 0)


def env_rank_world() -> tuple[int, int, int]:
    """(rank, local_rank, world_size) from the torchrun environment (1-process defaults otherwise)."""
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def make_sharded(env_id: str, total_envs: int, rank: int | None = None, world_size: int | None = None, **kwargs):
    """This rank's shard of a ``total_envs``-wide vector env (device = ``cuda:LOCAL_RANK`` unless given)."""
    from .registration import make_vec

    r, lr, w = env_rank_world()
    rank = r if rank is None else rank
    world_size = w if world_size is None else world_size
    start, count = shard_bounds(total_envs, world_size, rank)
    kwargs.setdefault("device", f"cuda:{lr}")
    return make_vec(env_id, num_envs=count, env_offset=start, **kwargs)


class BatchGather:
    """Gathers per-rank step outputs into one ``[total, ...]`` batch on every rank (``dst=None``) or on one rank.

    Equal shard sizes use ``all_gather_into_tensor`` (one NCCL call per tensor, written in place into the cached
    global batch); ragged shards are padded to the largest shard, gathered and compacted.
    """

    def __init__(self, total: int, world_size: int, rank: int, group=None, dst: int | None = None):
        self.total, self.world, self.rank, self.group, self.dst = int(total), world_size, rank, group, dst
        self.bounds = [shard_bounds(total, world_size, r) for r in range(world_size)]
        self.equal = len({c for _, c in self.bounds}) == 1
        self._buf: dict[str, torch.Tensor] = {}

    def _buffer(self, key: str, like: torch.Tensor) -> torch.Tensor:
        shape = (self.total,) + tuple(like.shape[1:])
        b = self._buf.get(key)
        if b is None or b.shape != shape or b.dtype != like.dtype or b.device != like.device:
            b = torch.empty(shape, dtype=like.dtype, device=like.device)
            self._buf[key] = b
        return b

    def __call__(self, **tensors: torch.Tensor) -> dict[str, torch.Tensor]:
        out = {}
        for key, t in tensors.items():
            if t.shape[0] != self.bounds[self.rank][1]:
                raise ValueError(f"{key}: leading dim {t.shape[0]} is not this rank's shard size {self.bounds[self.rank][1]}")
            as_u8 = t.dtype == torch.bool
            src = t.view(torch.uint8) if as_u8 else t
            full = self._buffer(key, src)
            src = src.contiguous()
            if self.equal and self.dst is not None:
                views = [full[s:s + c] for s, c in self.bounds] if self.rank == self.dst else None
                dist.gather(src, views, dst=self.dst, group=self.group)
            elif self.equal:
                dist.all_gather_into_tensor(full, src, group=self.group)
            else:  # ragged shards: pad every shard to the largest, gather, then compact into the global batch
                maxc = max(c for _, c in self.bounds)
                padded = torch.zeros((maxc,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
                padded[: src.shape[0]] = src
                stage = torch.empty((self.world * maxc,) + tuple(src.shape[1:]), dtype=src.dtype, device=src.device)
                dist.all_gather_into_tensor(stage, padded, group=self.group)
                for r, (s0, c) in enumerate(self.bounds):
                    full[s0:s0 + c] = stage[r * maxc:r * maxc + c]
            out[key] = full.view(torch.bool) if as_u8 else full
        return out


# ----------------------------------------------------------------------------------------------------------------------
def _np_dtype(dt):
    import numpy as np

    return np.dtype(np.bool_) if dt == torch.bool else torch.empty((), dtype=dt).numpy().dtype


class HostBatch:
    """ONE host-side batch shared by every rank of a node.

    ``depth`` slots, each holding the step outputs of ALL envs key by key -- ``obs [N_total, ...]``, ``reward [N_total]``,
    ... (struct-of-arrays keys such as Humanoid's ``info [13][n]`` become ``[13][N_total]``) -- in a shared-memory file that
    each rank maps and page-locks in its own CUDA context, so every GPU DMAs its shard's rows into place over its OWN PCIe
    link (8 links in parallel instead of a gather to rank 0 followed by one copy over rank 0's link).  It plays the role of
    ``AsyncVectorEnv``'s shared-memory observation buffer (gymnasium/vector/async_vector_env.py:234-245; the workers write
    their slice at :849-852).

    Header (one cache line per counter): ``seq[r]`` = number of steps whose rows rank r has landed (written by the GPU: an
    8-byte copy queued behind the data copies on the same stream; by the host in the CPU tests), ``ack`` = number of steps
    the consumer has released.  Step k lives in slot ``k % depth``; a producer may overwrite it once ``ack >= k-depth+1``.

    ``layout``: ``[(key, shape, torch dtype, ...)]`` of ONE shard's outputs (``B200VectorEnv.packed_outputs()[1]``);
    ``bounds``: ``[(start, count)]`` per rank (``shard_bounds``); ``soa_keys``: keys laid out ``[c][n]`` instead of ``[n][...]``.
    """

    LINE = 64

    def __init__(self, layout, bounds, rank: int, tag: str = "0", depth: int = 3, soa_keys=(), barrier=None,
                 register: bool = True, directory: str | None = None):
        import mmap

        import numpy as np

        self.world, self.rank, self.depth = len(bounds), int(rank), int(depth)
        self.bounds = [(int(s), int(c)) for s, c in bounds]
        self.total = sum(c for _, c in self.bounds)
        n_mine = self.bounds[self.rank][1]
        self.keys = []  # (key, global shape, numpy dtype, slot offset, row bytes, soa rows)
        off = 0
        for entry in layout:
            key, shape, dt = entry[0], tuple(entry[1]), entry[2]
            npdt = _np_dtype(dt)
            if key in soa_keys:
                if len(shape) != 2 or shape[1] != n_mine:
                    raise ValueError(f"{key}: a struct-of-arrays key must have shape (c, n), got {shape}")
                gshape, rowb, rows = (shape[0], self.total), npdt.itemsize, shape[0]
            else:
                if shape[0] != n_mine:
                    raise ValueError(f"{key}: leading dim {shape[0]} is not this rank's shard size {n_mine}")
                gshape, rowb, rows = (self.total,) + shape[1:], int(np.prod(shape[1:], dtype=np.int64)) * npdt.itemsize, 0
            self.keys.append((key, gshape, npdt, off, rowb, rows))
            off = (off + int(np.prod(gshape, dtype=np.int64)) * npdt.itemsize + 255) // 256 * 256
        self.slot_bytes = max(off, 256)
        # counters (one line per rank + the ack line), then per rank a line-aligned ring of sequence-word SOURCES for the
        # copy-engine landing (HostBatchPipeline's Python path): the value step k publishes is written there by the host and
        # copied behind the data by the same stream
        self.src_ring = 2 * self.depth + 2
        self._src_off = self.LINE * (self.world + 1)
        self._src_stride = (8 * self.src_ring + self.LINE - 1) // self.LINE * self.LINE
        self.header_bytes = (self._src_off + self._src_stride * self.world + 4095) // 4096 * 4096
        self.total_bytes = self.header_bytes + self.depth * self.slot_bytes
        if barrier is None:
            barrier = dist.barrier if (dist.is_available() and dist.is_initialized() and self.world > 1) else (lambda: None)
        name = f"b2e_hostbatch_{os.environ.get('MASTER_PORT', '0')}_{os.getuid()}_{tag}"
        self.path = os.path.join(directory or self._pick_dir(self.total_bytes), name)
        if rank == 0:
            try:
                os.unlink(self.path)
            except FileNotFoundError:
                pass
            fd = os.open(self.path, os.O_CREAT | os.O_RDWR | os.O_EXCL, 0o600)
            os.ftruncate(fd, self.total_bytes)
            barrier()
        else:
            barrier()
            fd = os.open(self.path, os.O_RDWR)
        self._mm = mmap.mmap(fd, self.total_bytes)
        os.close(fd)
        barrier()  # everybody has it mapped: the name can go (the pages live as long as a mapping does)
        if rank == 0:
            os.unlink(self.path)
        self._np = np.frombuffer(self._mm, dtype=np.uint8)
        self._hdr = self._np[: self.header_bytes].view(np.int64)
        self._addr = self._np.ctypes.data
        self._registered = False
        self._views: dict = {}
        # first touch decides the NUMA node of a page: every rank faults in ITS rows (the pages its GPU will write), rank 0 the
        # header -- before anybody page-locks the buffer
        if rank == 0:
            self._np[: self.header_bytes] = 0
        start, count = self.bounds[self.rank]
        for j in range(self.depth):
            for key, arr in self.views(j).items():
                if key in soa_keys:
                    arr[:, start:start + count] = 0
                else:
                    arr[start:start + count] = 0
        barrier()
        if register:
            from . import _lib

            self._lib = _lib.load()
            _lib.check(self._lib.b2e_host_register(self._addr, self.total_bytes), "b2e_host_register")
            self._registered = True
        barrier()

    @staticmethod
    def _pick_dir(nbytes: int) -> str:
        for d in (os.environ.get("B2E_HOSTBATCH_DIR"), "/dev/shm", "/tmp"):
            if d and os.path.isdir(d):
                try:
                    st = os.statvfs(d)
                    if st.f_bavail * st.f_frsize > nbytes + (64 << 20):
                        return d
                except OSError:
                    continue
        return "/tmp"

    # ---- addressing ------------------------------------------------------------------------------------------------
    def views(self, k: int) -> dict:
        """numpy views ``{key: global array}`` of the slot step k lives in."""
        import numpy as np

        j = k % self.depth
        hit = self._views.get(j)
        if hit is not None:
            return hit
        base = self.header_bytes + j * self.slot_bytes
        out = {}
        for key, gshape, npdt, off, _rowb, _rows in self.keys:
            nb = int(np.prod(gshape, dtype=np.int64)) * npdt.itemsize
            out[key] = self._np[base + off: base + off + nb].view(npdt).reshape(gshape)
        self._views[j] = out
        return out

    def segments(self, k: int, src_rank: int, dev_ptrs: dict) -> list[tuple]:
        """Copy segments ``(host_dst, dev_src, dst_pitch, src_pitch, width, height)`` that land rank `src_rank`'s shard of
        step k: one contiguous run per row-major key, one pitched copy per struct-of-arrays key."""
        base = self._addr + self.header_bytes + (k % self.depth) * self.slot_bytes
        start, count = self.bounds[src_rank]
        segs = []
        for key, _gshape, npdt, off, rowb, rows in self.keys:
            if rows:
                w = count * npdt.itemsize
                segs.append((base + off + start * npdt.itemsize, dev_ptrs[key], self.total * npdt.itemsize, w, w, rows))
            else:
                segs.append((base + off + start * rowb, dev_ptrs[key], 0, 0, count * rowb, 1))
        return segs

    def seq_addr(self, rank: int | None = None) -> int:
        r = self.rank if rank is None else rank
        return self._addr + r * self.LINE

    def seq_source(self, k: int) -> int:
        """Writes k+1 into this rank's source ring and returns its address (the last copy segment of step k reads it)."""
        i = (self._src_off + self._src_stride * self.rank) // 8 + k % self.src_ring
        self._hdr[i] = k + 1
        return self._addr + 8 * i

    # ---- protocol --------------------------------------------------------------------------------------------------
    def _seq(self, r: int) -> int:
        return int(self._hdr[r * self.LINE // 8])

    def acked(self) -> int:
        return int(self._hdr[self.world * self.LINE // 8])

    def publish_host(self, k: int) -> None:
        """Host-side publication of step k (CPU tests; on a GPU the copy stream writes the counter itself)."""
        self._hdr[self.rank * self.LINE // 8] = k + 1

    def wait_writable(self, k: int, timeout: float = 120.0) -> None:
        """Blocks until the slot of step k has been released by the consumer (always true for the first `depth` steps)."""
        need = k - self.depth + 1
        if need <= 0 or self.acked() >= need:
            return
        self._spin(lambda: self.acked() >= need, timeout, f"ack of step {need - 1}")

    def wait_ready(self, k: int, ranks=None, timeout: float = 120.0) -> dict:
        """Consumer: blocks until the rows of step k from every rank (or from `ranks`) have landed; returns `views(k)`."""
        ranks = range(self.world) if ranks is None else ranks
        if not all(self._seq(r) > k for r in ranks):
            self._spin(lambda: all(self._seq(r) > k for r in ranks), timeout, f"step {k} from ranks {list(ranks)}")
        return self.views(k)

    def ack(self, k: int) -> None:
        self._hdr[self.world * self.LINE // 8] = k + 1

    @staticmethod
    def _spin(cond, timeout, what):
        import time

        t0 = time.perf_counter()
        spins = 0
        while not cond():
            spins += 1
            if spins > 2000:
                time.sleep(0)  # yield: several ranks may share a core in a small container
                if time.perf_counter() - t0 > timeout:
                    raise TimeoutError(f"HostBatch: timed out waiting for {what}")

    def close(self) -> None:
        if self._registered:
            self._lib.b2e_host_unregister(self._addr)
            self._registered = False
        self._hdr = self._np = None
        self._views = {}
        try:
            self._mm.close()
        except (BufferError, ValueError):
            pass


class _CallRecorder:
    """Stands in for the ctypes library while a family's ``_step_kernel`` runs: instead of launching, every ``b2e_*`` call is
    recorded as (function address, machine-word arguments) -- what ``b2e_pipe_submit`` replays from C."""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        import ctypes as C

        fn = getattr(self._lib, name)
        if not name.startswith("b2e_"):
            return fn

        def record(*args):
            words = []
            for a in args:
                if a is None:
                    words.append(0)
                elif isinstance(a, int):
                    words.append(a & ((1 << 64) - 1))
                elif hasattr(a, "_obj"):  # ctypes.byref(struct): the struct lives as long as the env does
                    words.append(C.addressof(a._obj))
                elif isinstance(a, C._SimpleCData):
                    words.append(int(a.value or 0))
                elif isinstance(a, float):
                    raise TypeError(f"{name}: floating-point arguments cannot be replayed as machine words")
                else:
                    words.append(C.cast(a, C.c_void_p).value or 0)
            if len(words) > 16:
                raise TypeError(f"{name}: more than 16 arguments")
            self.calls.append((C.cast(fn, C.c_void_p).value, words))
            return 0

        return record


class HostBatchPipeline:
    """Pipelined end-to-end stepping of one shard.  ``submit(host_actions)`` enqueues the pinned H2D copy of the actions and
    the fused step launch on the caller's stream and, on a copy stream, the landing of the step outputs into this rank's
    rows of the shared :class:`HostBatch` followed by its 8-byte sequence word -- no host synchronisation.  The fast path
    (numpy-parity RNG) lands them with one kernel; the Python path (``fast=False``) with the copy engine.  ``consume(k)``
    (consumer rank) waits until every rank's rows of step k have landed and returns numpy views of the whole batch.  The
    copies of step k overlap the kernel of step k+1 (the env rotates over `depth` output buffers).

    ``mode="nccl"`` gathers the packed outputs of all ranks to the consumer with ONE NCCL gather on the side stream (NVLink),
    overlapped with the next step the same way; the consumer alone copies the gathered shards to the host (one PCIe link).
    """

    def __init__(self, env, world_size: int, rank: int, total_envs: int | None = None, tag: str = "0", depth: int = 3,
                 mode: str = "dma", consumer: int = 0, fast: bool = True):
        if env.output != "torch" or env.copy or env.out_buffers < depth:
            raise ValueError("HostBatchPipeline needs an env made with output='torch', copy=False, out_buffers >= depth")
        if mode not in ("dma", "nccl"):
            raise ValueError(f"mode must be 'dma' or 'nccl', got {mode!r}")
        import ctypes as C

        from . import _lib

        self.env, self.world, self.rank, self.depth, self.mode, self.consumer = env, world_size, rank, depth, mode, consumer
        self._C, self._lib_mod, self._lib = C, _lib, _lib.load()
        dev = env.device
        total = env.num_envs * world_size if total_envs is None else int(total_envs)
        bounds = [shard_bounds(total, world_size, r) for r in range(world_size)]
        if bounds[rank][1] != env.num_envs:
            raise ValueError(f"env has {env.num_envs} sub-envs but rank {rank}'s shard of {total} is {bounds[rank][1]}")
        self.is_consumer = rank == consumer
        self._rings = [env._outputs() for _ in range(env.out_buffers)]  # allocates the ring; the layout is fixed now
        wire, layout = env.packed_outputs()
        self.layout, self.wire_bytes = layout, int(wire.numel())
        soa = tuple(getattr(env, "soa_output_keys", ()))
        if mode == "dma":
            self.host = HostBatch(layout, bounds, rank, tag=f"{tag}_dma", depth=depth, soa_keys=soa)
        else:
            if len({c for _, c in bounds}) != 1:
                raise ValueError("mode='nccl' needs equal shards")
            # private to the consumer: nobody else writes it, so its "world" for the seq/ack protocol is 1 rank
            self.host = (HostBatch(layout, bounds, rank, tag=f"{tag}_nccl", depth=depth, soa_keys=soa, barrier=lambda: None)
                         if self.is_consumer else None)
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.k = 0
        self._ev_step = [torch.cuda.Event() for _ in range(depth)]
        self._ev_copy = [None] * depth
        self._cs_handle = self.copy_stream.cuda_stream
        self._seq_dev = torch.zeros(2 * depth + 2, dtype=torch.int64, device=dev)
        self._gathered = ([torch.empty((world_size, self.wire_bytes), dtype=torch.uint8, device=dev) for _ in range(depth)]
                          if mode == "nccl" and self.is_consumer else None)
        self._seg_cache: dict = {}
        # fast path (mode 'dma', numpy-parity RNG): the whole submit is ONE C call, b2e_pipe_submit, replaying the family's
        # recorded step call(s) -- set up lazily at the first submit, when the action dtype / shape is known
        self._fast = None if (mode == "dma" and fast and env.rng_mode == "numpy") else False
        self._slots = None
        # the fast path lands a step's rows with one kernel launch (SM stores over PCIe, then the sequence word); the copy
        # engine's per-key copies, alone or as one CUDA graph, were slower (DESIGN.md section 6)
        self.landing = "kernel"
        self._pinned_ptrs: set = set()
        self._pinned_keep: list = []

    def pinned_actions(self, count: int = 1, dtype=None) -> list:
        """`count` page-locked numpy arrays shaped like one step's action batch.  ``submit`` DMAs straight from an array
        obtained here (no staging copy); the caller must leave it untouched until that step has been consumed."""
        import numpy as np

        env = self.env
        if dtype is None:
            dtype = np.int64 if env.discrete_actions else np.float32
        shape = (env.num_envs,) if env.discrete_actions else (env.num_envs,) + tuple(env.single_action_space.shape)
        out = []
        for _ in range(count):
            t = torch.from_numpy(np.zeros(shape, dtype=dtype)).pin_memory()
            a = t.numpy()
            self._pinned_keep.append(t)
            self._pinned_ptrs.add(a.ctypes.data)
            out.append(a)
        return out

    def _segments(self, k: int, out: dict):
        """ctypes array of the copy segments of step k (cached per (slot, output set))."""
        key = (k % self.depth, out["_wire"].data_ptr())
        hit = self._seg_cache.get(key)
        if hit is not None:
            return hit
        segs = []
        if self.mode == "dma":
            segs += self.host.segments(k, self.rank, {e[0]: out[e[0]].data_ptr() for e in self.layout})
        else:
            g = self._gathered[k % self.depth]
            for r in range(self.world):
                base = g[r].data_ptr()
                segs += self.host.segments(k, r, {e[0]: base + e[3] for e in self.layout})
        # publication: the sequence word goes pinned source -> device scratch -> seq word, two DMAs queued behind the data (a
        # host->host cudaMemcpyAsync is NOT stream-ordered: the runtime copies on the calling thread, ahead of the data)
        bounce = self._seq_dev[k % self._seq_dev.numel():].data_ptr()
        segs.append((bounce, 0, 0, 0, 8, 1))  # source patched per step: HostBatch.seq_source(k)
        segs.append((self.host.seq_addr(), bounce, 0, 0, 8, 1))
        arr = (self._lib_mod.CopySeg * len(segs))(*[self._lib_mod.CopySeg(*s) for s in segs])
        self._seg_cache[key] = (arr, len(segs))
        return self._seg_cache[key]

    def _setup_fast(self, a) -> bool:
        """Builds the b2e_pipe_slot of every (staging buffer, output set, landing slot) triple for host actions shaped and
        typed like `a`.  Returns False (slow path) if the family's step cannot be replayed from C."""
        import numpy as np

        C, L = self._C, self._lib_mod
        env, dev, depth = self.env, self.env.device, self.depth
        if not isinstance(a, np.ndarray) or a.shape[0] != env.num_envs or a.dtype.kind not in "iuf":
            return False
        if not getattr(env, "replayable_step", True):  # the family's step is more than C-ABI calls (e.g. Taxi's fickle passenger)
            return False
        if env.discrete_actions and (a.ndim != 1 or a.dtype not in (np.int64, np.int32, np.uint8)):
            return False
        if not env.discrete_actions and a.dtype not in (np.float32, np.float64):
            return False
        from .vector_env import _ACT_DTYPES

        self._fast_shape, self._fast_dtype = a.shape, a.dtype
        self._main_handle = torch.cuda.current_stream(dev).cuda_stream
        self._keep = []  # buffers the slots point into
        slots = (L.PipeSlot * depth)()
        for j in range(depth):
            out = self._rings[j]
            staging = torch.from_numpy(np.empty(a.shape, dtype=a.dtype)).pin_memory()
            act_dev = torch.empty(a.shape, dtype=staging.dtype, device=dev)
            rec = _CallRecorder(env._lib)
            real = env._lib
            env._batch.action_dtype = _ACT_DTYPES[act_dev.dtype]
            env._lib = rec
            try:
                with torch.cuda.device(dev):
                    env._step_kernel(act_dev, out)
            except TypeError:
                return False
            finally:
                env._lib = real
            if not rec.calls:
                return False
            calls = (L.Call * len(rec.calls))()
            for c, (fn, words) in zip(calls, rec.calls):
                c.fn, c.nargs = fn, len(words)
                for i, wd in enumerate(words):
                    c.args[i] = wd
            seg_list = self.host.segments(j, self.rank, {e[0]: out[e[0]].data_ptr() for e in self.layout})
            # the two publication segments of the copy-engine path: the landing kernel stores the sequence word itself and
            # takes only its address from the last one
            bounce = self._seq_dev[j:].data_ptr()
            seg_list.append((bounce, 0, 0, 0, 8, 1))
            seg_list.append((self.host.seq_addr(), bounce, 0, 0, 8, 1))
            segs = (L.CopySeg * len(seg_list))(*[L.CopySeg(*sg) for sg in seg_list])
            sl = slots[j]
            sl.staging_host, sl.actions_dev, sl.action_bytes = staging.data_ptr(), act_dev.data_ptr(), a.nbytes
            sl.calls, sl.ncalls = calls, len(rec.calls)
            sl.segs, sl.nsegs = segs, len(seg_list)
            L.check(self._lib.b2e_pipe_slot_init(C.byref(sl)), "b2e_pipe_slot_init")
            L.check(self._lib.b2e_pipe_slot_land_kernel(C.byref(sl)), "b2e_pipe_slot_land_kernel")
            self._keep += [staging, act_dev, calls, segs]
        self._slots = slots
        self._ack_addr = self.host._addr + self.host.world * self.host.LINE
        return True

    def submit(self, actions) -> int:
        if self._fast is None:
            if not self.env._has_reset:
                from . import errors

                raise errors.ResetNeeded("Cannot call env.step() before calling env.reset()")
            self._fast = self._setup_fast(actions)
        if self._fast:
            a = actions
            if getattr(a, "shape", None) != self._fast_shape or a.dtype != self._fast_dtype or not a.flags.c_contiguous:
                import numpy as np

                a = np.ascontiguousarray(actions, dtype=self._fast_dtype)
                if a.shape != self._fast_shape:
                    raise ValueError(f"expected actions of shape {self._fast_shape}, got {a.shape}")
            k, j = self.k, self.k % self.depth
            ptr = a.ctypes.data
            st = self._lib.b2e_pipe_submit(self._C.byref(self._slots[j]), ptr, self._main_handle, self._cs_handle,
                                           self._ack_addr, k - self.depth + 1, k + 1,
                                           1 if ptr in self._pinned_ptrs else 0, 120.0)
            if st:
                self._lib_mod.check(st, "b2e_pipe_submit")
            self.env._out = self._rings[j]
            self.k += 1
            return k
        k, j = self.k, self.k % self.depth
        env, dev = self.env, self.env.device
        main = torch.cuda.current_stream(dev)
        if self._ev_copy[j] is not None:
            main.wait_event(self._ev_copy[j])  # the kernel of step k re-uses the output set step k-depth was copied from
        env.step(actions)
        out = env._out
        self._ev_step[j].record(main)
        cs = self.copy_stream
        cs.wait_event(self._ev_step[j])
        if self.mode == "nccl":
            with torch.cuda.stream(cs):
                dst = list(self._gathered[j].unbind(0)) if self.is_consumer else None
                dist.gather(out["_wire"], dst, dst=self.consumer)
        if self.host is not None:
            self.host.wait_writable(k)
            arr, cnt = self._segments(k, out)
            arr[cnt - 2].dev_src = self.host.seq_source(k)
            st = self._lib.b2e_copy_to_host_async(arr, cnt, self._cs_handle)
            if st:
                self._lib_mod.check(st, "b2e_copy_to_host_async")
        ev = self._ev_copy[j] or torch.cuda.Event()
        ev.record(cs)
        self._ev_copy[j] = ev
        self.k += 1
        return k

    def consume(self, k: int, ack: bool = True) -> dict:
        """Consumer rank: numpy views ``{key: [N_total, ...]}`` of step k's batch.  With ``ack=True`` the slot is released to
        the producers at once -- the views may then be overwritten as soon as `depth - 1` further steps have been submitted
        (a fast producer rank can be that far ahead), so read them first or pass ``ack=False`` and call :meth:`release`
        when done with them."""
        ranks = None if self.mode == "dma" else [self.rank]
        out = self.host.wait_ready(k, ranks=ranks)
        if ack:
            self.host.ack(k)
        return out

    def release(self, k: int) -> None:
        """Consumer rank: hands the slot of step k back to the producers (after ``consume(k, ack=False)``)."""
        self.host.ack(k)

    def drain(self) -> None:
        self.copy_stream.synchronize()

    def close(self) -> None:
        self.drain()
        if self._slots is not None:
            torch.cuda.synchronize(self.env.device)
            for sl in self._slots:
                self._lib.b2e_pipe_slot_destroy(self._C.byref(sl))
            self._slots = None
        if self.host is not None:
            self.host.close()
