"""Host-to-device ceiling of ONE host with N GPUs copying at the same time (round-1 review, item 4): what do N concurrent pinned
copies get per GPU, and does the kind of host memory change it?  Launch like the bench:
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29531 tools/h2d_probe.py
Every rank copies a 1 GiB host buffer to its own GPU, all ranks behind a barrier, three repetitions, CUDA events on the copy
stream(s); the line shows the SLOWEST rank's best repetition (GB/s per GPU) and N times that (aggregate).
Variants: cudaHostAlloc (what swtpg_alloc_pinned returns), the same split over 2 and 4 streams, write-combined, a
transparent-huge-page region registered with cudaHostRegister, and a hugetlbfs (2 MB pages, MAP_HUGETLB) region registered the
same way (it uses the 2 MB pages the host has reserved already; without them its mmap fails and the line says so).
CUDA runtime through ctypes (no torch tensors involved: torch would route an unknown host pointer through its pageable path)."""
import ctypes as C
import mmap
import os
import sys
import time

import torch.distributed as dist

rt = C.CDLL("libcudart.so.12")
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
if world > 1:
    dist.init_process_group("gloo")
SIZE = 1 << 30
MAP_HUGETLB, MADV_HUGEPAGE = 0x40000, 14
libc = C.CDLL("libc.so.6", use_errno=True)


def ck(e, what):
    if e != 0:
        raise RuntimeError(f"{what}: cuda error {e}")


def barrier():
    if world > 1:
        dist.barrier()


def max_all(x):
    if world == 1:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


ck(rt.cudaSetDevice(local), "cudaSetDevice")
dev = C.c_void_p()
ck(rt.cudaMalloc(C.byref(dev), C.c_size_t(SIZE)), "cudaMalloc")
streams = []
for _ in range(4):
    s = C.c_void_p()
    ck(rt.cudaStreamCreateWithFlags(C.byref(s), 1), "stream")
    streams.append(s)
ev = []
for _ in range(2):
    e = C.c_void_p()
    ck(rt.cudaEventCreate(C.byref(e)), "event")
    ev.append(e)


def timed(host_ptr, n_streams):
    """best of 3: ms for SIZE bytes split evenly over n_streams streams, everything started behind a barrier"""
    best = 1e30
    part = SIZE // n_streams
    for _ in range(4):
        ck(rt.cudaDeviceSynchronize(), "sync")
        barrier()
        t0 = time.perf_counter()
        for i in range(n_streams):
            ck(rt.cudaMemcpyAsync(C.c_void_p(dev.value + i * part), C.c_void_p(host_ptr + i * part), C.c_size_t(part), 1, streams[i]), "memcpy")
        ck(rt.cudaDeviceSynchronize(), "sync")
        best = min(best, (time.perf_counter() - t0) * 1e3)
    return best


def report(name, ms, note=""):
    slow = max_all(ms)
    if rank == 0:
        gbs = SIZE / slow / 1e6
        print(f"{name:46s} {gbs:7.2f} GB/s per GPU (slowest of {world})  {gbs * world:8.1f} GB/s aggregate  {note}", flush=True)


def touch(ptr):
    C.memset(C.c_void_p(ptr), 1, SIZE)


if rank == 0:
    print(f"== h2d_probe: {world} rank(s), {SIZE >> 20} MiB per rank per copy, host cores {os.cpu_count()}", flush=True)
    for f in ("/sys/kernel/mm/transparent_hugepage/enabled", "/proc/sys/vm/nr_hugepages"):
        try:
            print(f"   {f}: {open(f).read().strip()}", flush=True)
        except OSError as e:
            print(f"   {f}: {e}", flush=True)

# 1. cudaHostAlloc, 1 / 2 / 4 streams
p = C.c_void_p()
ck(rt.cudaHostAlloc(C.byref(p), C.c_size_t(SIZE), 1), "cudaHostAlloc")
touch(p.value)
for n in (1, 2, 4):
    report(f"cudaHostAlloc, {n} stream(s)", timed(p.value, n))
rt.cudaFreeHost(p)

# 2. write-combined
p = C.c_void_p()
ck(rt.cudaHostAlloc(C.byref(p), C.c_size_t(SIZE), 1 | 4), "cudaHostAlloc wc")
touch(p.value)
report("cudaHostAlloc write-combined, 1 stream", timed(p.value, 1))
rt.cudaFreeHost(p)


def registered(name, flags, advise):
    try:
        mm = mmap.mmap(-1, SIZE + (2 << 20), flags=mmap.MAP_PRIVATE | mmap.MAP_ANONYMOUS | flags)
    except (OSError, ValueError) as e:
        report(name, 1e30, f"mmap failed on this rank: {e}")
        return
    base = C.addressof(C.c_char.from_buffer(mm))
    ptr = (base + (2 << 20) - 1) & ~((2 << 20) - 1)
    if advise:
        libc.madvise(C.c_void_p(ptr), C.c_size_t(SIZE), MADV_HUGEPAGE)
    touch(ptr)
    huge = ""
    if advise:
        try:
            for line in open("/proc/self/smaps_rollup"):
                if line.startswith("AnonHugePages"):
                    huge = "AnonHugePages " + line.split(":")[1].strip()
        except OSError:
            pass
    e = rt.cudaHostRegister(C.c_void_p(ptr), C.c_size_t(SIZE), 1)
    if e != 0:
        rt.cudaGetLastError()
        report(name, 1e30, f"cudaHostRegister failed ({e})")
        return
    report(name, timed(ptr, 1), huge)
    rt.cudaHostUnregister(C.c_void_p(ptr))


registered("4 KB pages + cudaHostRegister", 0, False)
registered("transparent huge pages + cudaHostRegister", 0, True)
barrier()
registered("hugetlbfs 2 MB pages + cudaHostRegister", MAP_HUGETLB, False)
barrier()
if world > 1:
    dist.destroy_process_group()
