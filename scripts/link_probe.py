"""Raw host-link probe for the single host-side batch (no env, no kernels): every rank copies `--mb` MB device -> host
`--iters` times, all ranks at once, into (a) its own cudaHostAlloc buffer, (b) its slice of ONE shared-memory file first
touched by rank 0 (what HostBatch does), (c) the same with every rank touching its own slice first.  Prints per-rank and
aggregate GB/s (CUDA events, max over ranks) -- the ceiling `e2e` of a microsecond-kernel family can reach at this world size.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 scripts/link_probe.py
"""
import argparse
import mmap
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gymnasium_b200 import _lib  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=float, default=1.625)  # CartPole-v1 at 65536 envs: 26 B/env
    ap.add_argument("--h2d-mb", type=float, default=0.5)
    ap.add_argument("--iters", type=int, default=400)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    nb = int(args.mb * (1 << 20)) // 256 * 256
    hb = int(args.h2d_mb * (1 << 20)) // 256 * 256
    src = torch.empty(nb, dtype=torch.uint8, device=dev).random_(0, 255)
    act_dev = torch.empty(hb, dtype=torch.uint8, device=dev)
    act_host = torch.empty(hb, dtype=torch.uint8).pin_memory()
    s_out, s_in = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def shared(tag, owner_touch):
        path = f"/dev/shm/b2e_probe_{os.environ.get('MASTER_PORT', '0')}_{tag}"
        total = nb * world
        if rank == 0:
            fd = os.open(path, os.O_CREAT | os.O_RDWR | os.O_TRUNC, 0o600)
            os.ftruncate(fd, total)
            barrier()
        else:
            barrier()
            fd = os.open(path, os.O_RDWR)
        mm = mmap.mmap(fd, total)
        os.close(fd)
        arr = np.frombuffer(mm, dtype=np.uint8)
        if owner_touch:
            arr[rank * nb:(rank + 1) * nb] = 0
        elif rank == 0:
            arr[:] = 0
        barrier()
        if rank == 0:
            os.unlink(path)
        _lib.check(lib.b2e_host_register(arr.ctypes.data, total), "b2e_host_register")
        return mm, arr, arr.ctypes.data + rank * nb

    def timed(dst_ptr, duplex):
        import ctypes as C

        seg = (_lib.CopySeg * 1)()
        seg[0].host_dst, seg[0].dev_src, seg[0].dst_pitch, seg[0].src_pitch, seg[0].width, seg[0].height = dst_ptr, src.data_ptr(), 0, 0, nb, 1
        best = None
        for rep in range(3):
            torch.cuda.synchronize()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s_out):
                e0.record()
                for _ in range(args.iters):
                    _lib.check(lib.b2e_copy_to_host_async(seg, 1, C.c_void_p(s_out.cuda_stream)), "copy")
                e1.record()
            if duplex:
                with torch.cuda.stream(s_in):
                    for _ in range(args.iters):
                        act_dev.copy_(act_host, non_blocking=True)
            torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t = float(t.item())
            best = t if best is None else min(best, t)
        return best

    rows = []
    pinned = torch.empty(nb, dtype=torch.uint8).pin_memory()
    for name, make in (("cudaHostAlloc per rank", lambda: (None, None, pinned.data_ptr())),
                       ("shared file, rank 0 touches", lambda: shared("a", False)),
                       ("shared file, owner touches", lambda: shared("b", True))):
        mm, arr, ptr = make()
        for duplex in (False, True):
            t = timed(ptr, duplex)
            rows.append((name, duplex, t))
            if rank == 0:
                per = nb * args.iters / t / 1e9
                print(f"world={world} {name:30s} {'D2H+H2D' if duplex else 'D2H only':9s}: {t / args.iters * 1e6:7.1f} us per "
                      f"{nb / 1e6:.2f} MB copy, {per:5.1f} GB/s per rank, {per * world:6.1f} GB/s aggregate", flush=True)
        if arr is not None:
            lib.b2e_host_unregister(arr.ctypes.data)
    # the landing kernel (SM stores into the mapped shared file + sequence word)
    import ctypes as C

    mm, arr, ptr = shared("c", False)
    seq_mm = mmap.mmap(-1, 4096)
    seq_np = np.frombuffer(seq_mm, dtype=np.int64)
    _lib.check(lib.b2e_host_register(seq_np.ctypes.data, 4096), "b2e_host_register")
    seg = (_lib.CopySeg * 1)()
    seg[0].host_dst, seg[0].dev_src, seg[0].dst_pitch, seg[0].src_pitch, seg[0].width, seg[0].height = ptr, src.data_ptr(), 0, 0, nb, 1
    plan = C.c_void_p()
    _lib.check(lib.b2e_land_plan_create(seg, 1, seq_np.ctypes.data, C.byref(plan)), "b2e_land_plan_create")
    best = None
    for rep in range(3):
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(s_out):
            e0.record()
            for i in range(args.iters):
                lib.b2e_land_plan_launch(plan, i + 1, C.c_void_p(s_out.cuda_stream))
            e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = float(t.item()) if best is None else min(best, float(t.item()))
    ok = int(seq_np[0]) == args.iters and bool((arr[rank * nb:(rank + 1) * nb] == src.cpu().numpy()).all())
    if rank == 0:
        per = nb * args.iters / best / 1e9
        print(f"world={world} landing kernel                     : {best / args.iters * 1e6:7.1f} us per {nb / 1e6:.2f} MB, "
              f"{per:5.1f} GB/s per rank, {per * world:6.1f} GB/s aggregate, data+seq {'ok' if ok else 'WRONG'}", flush=True)
    lib.b2e_land_plan_destroy(plan)
    lib.b2e_host_unregister(arr.ctypes.data)
    lib.b2e_host_unregister(seq_np.ctypes.data)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
