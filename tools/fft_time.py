"""times batched rfft of one order: python tools/fft_time.py ORDER"""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as entry
order = int(sys.argv[1]); pkg = entry.load_package(); pkg.set_device(0)
n = 1 << order; batch = (1 << 28) // n
x = torch.rand((batch, n), device="cuda") * 2 - 1
plan = pkg.RFFTPlan(order, "float32"); plan.set_stream(torch.cuda.current_stream())
spec = torch.empty((batch, n // 2 + 1), dtype=torch.complex64, device="cuda")
for _ in range(3): plan.rfft(x, out=spec)
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(10): plan.rfft(x, out=spec)
b.record(); torch.cuda.synchronize()
ms = a.elapsed_time(b) / 10
print(f"order {order}: {ms*1e3:.0f} us, {batch*(4*n+8*(n//2+1))/ms/1e6:.0f} GB/s")
