"""Does a device->host copy overlap a running kernel on this box?  (The chunked copy pipeline mtfjsp_step_host_packed
used before its kernel wrote the records into mapped host memory assumed it did.)  A ~100 us memory-bound kernel on one
stream, a 4.7 MB pinned D2H copy on another."""
import time

import torch

dev = torch.device("cuda")
x = torch.empty(200 * 1024 * 1024 // 4, device=dev)           # 200 MB: x.mul_ reads + writes 400 MB
d = torch.empty(4718592, dtype=torch.uint8, device=dev)
h = torch.empty(4718592, dtype=torch.uint8).pin_memory()
s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()


def t(fn, n=30):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        fn()
        torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e6


def kern():
    with torch.cuda.stream(s1):
        x.mul_(1.0001)


def copy():
    with torch.cuda.stream(s2):
        h.copy_(d, non_blocking=True)


def both():
    kern(); copy()


def serial():
    with torch.cuda.stream(s1):
        x.mul_(1.0001)
        h.copy_(d, non_blocking=True)


print("kernel alone %.1f us, copy alone %.1f us, both on two streams %.1f us, same stream %.1f us" % (t(kern), t(copy), t(both), t(serial)))
