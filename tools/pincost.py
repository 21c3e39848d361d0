# what page-locking host memory costs on this box: cudaHostAlloc / cudaFreeHost of 16 and 128 MiB, and a pageable against a
# page-locked H2D copy of 64 MiB (the numbers behind the stream shim's buffer policy, zs_stream.cu: HostBuf / BufPool)
import ctypes, time, torch
rt = ctypes.CDLL("libcudart.so.12")
torch.cuda.init(); torch.zeros(1, device="cuda")
for mib in (16, 128):
    p = ctypes.c_void_p()
    t0 = time.perf_counter(); rc = rt.cudaHostAlloc(ctypes.byref(p), ctypes.c_size_t(mib << 20), 1); t1 = time.perf_counter()
    rt.cudaFreeHost(p); t2 = time.perf_counter()
    print(f"cudaHostAlloc {mib} MiB: {1e3 * (t1 - t0):.2f} ms (rc {rc}), cudaFreeHost {1e3 * (t2 - t1):.2f} ms")
n = 64 << 20
d = torch.empty(n, dtype=torch.uint8, device="cuda")
for name, h in (("pageable (fresh)", torch.empty(n, dtype=torch.uint8)), ("page-locked", torch.empty(n, dtype=torch.uint8).pin_memory())):
    for rep in range(3):
        torch.cuda.synchronize(); t0 = time.perf_counter(); d.copy_(h); torch.cuda.synchronize()
        print(f"H2D 64 MiB {name}, pass {rep}: {1e3 * (time.perf_counter() - t0):.2f} ms")
    for rep in range(2):
        torch.cuda.synchronize(); t0 = time.perf_counter(); h.copy_(d); torch.cuda.synchronize()
        print(f"D2H 64 MiB {name}, pass {rep}: {1e3 * (time.perf_counter() - t0):.2f} ms")
