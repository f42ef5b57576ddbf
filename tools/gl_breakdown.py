"""Time the two Griffin-Lim kernels separately on the cfg3 shape (scratch measurement tool)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import spev_tts_b200 as sp
from spev_tts_b200 import _lib
dev = torch.device("cuda", 0)
B, T = int(sys.argv[1]) if len(sys.argv) > 1 else 16, int(sys.argv[2]) if len(sys.argv) > 2 else 800
ctx = sp.Context.get(dev, fmin=0.0, fmax=8000.0)
fb = sp.make_batch(ctx, n_frames=[T] * B, with_chunks=True)
F = fb.n_frames
g = torch.Generator(device=dev).manual_seed(0)
ang = torch.randn(F, 520, 2, generator=g, device=dev).contiguous()
tprev = torch.randn(F, 520, 2, generator=g, device=dev).contiguous()
S = torch.rand(F, 520, generator=g, device=dev)
y = torch.zeros(fb.n_out_samples, device=dev)
st = torch.cuda.current_stream(dev).cuda_stream
lib = ctx.lib
def t_loop(fn, n=60, reps=5):
    for _ in range(2): 
        for _ in range(n): fn()
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(reps):
        a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n): fn()
        b.record(); torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) / n * 1e3)
    return best
k4 = t_loop(lambda: lib.spev_istft(ctx.handle, fb.desc, ang.data_ptr(), 520, y.data_ptr(), st))
k5 = t_loop(lambda: lib.spev_gl_phase_update(ctx.handle, fb.desc, y.data_ptr(), S.data_ptr(), 520, ang.data_ptr(), tprev.data_ptr(), 520, 0.4975, 1, st))
k5n = t_loop(lambda: lib.spev_gl_phase_update(ctx.handle, fb.desc, y.data_ptr(), S.data_ptr(), 520, ang.data_ptr(), tprev.data_ptr(), 520, 0.4975, 0, st))
k5s = t_loop(lambda: lib.spev_stft(ctx.handle, fb.desc, y.data_ptr(), ang.data_ptr(), 520, st))
def both():
    lib.spev_istft(ctx.handle, fb.desc, ang.data_ptr(), 520, y.data_ptr(), st)
    lib.spev_gl_phase_update(ctx.handle, fb.desc, y.data_ptr(), S.data_ptr(), 520, ang.data_ptr(), tprev.data_ptr(), 520, 0.4975, 1, st)
kb = t_loop(both)
# the real thing: spev_griffinlim (tickets + PDL chain), 60 iterations
ws = torch.empty(lib.spev_griffinlim_workspace_bytes(F), dtype=torch.uint8, device=dev)
def full():
    _lib.check(lib.spev_griffinlim(ctx.handle, fb.desc, S.data_ptr(), 520, None, 7, 60, 0.99, y.data_ptr(), ws.data_ptr(), ws.numel(), st))
kf = t_loop(full, n=1, reps=8)
print(f"B={B} T={T} frames={F} ftiles={fb.n_ftiles} ctiles={fb.n_ctiles}")
print(f"spev_griffinlim 60 it: {kf/1e3:8.3f} ms  -> {kf/60:6.2f} us/iter  roofline {F*(20516*60+5128)/kf/1e3/6542.1:.3f}")
print(f"istft          {k4:8.2f} us/launch   {F*(4104+1024)/k4/1e3:8.1f} GB/s")
print(f"phase_update   {k5:8.2f} us/launch   {F*15388/k5/1e3:8.1f} GB/s")
print(f"phase no-prev   {k5n:8.2f} us/launch   (no tprev loads: S 2 KB read, ang+tprev 8 KB written per frame)")
print(f"stft only      {k5s:8.2f} us/launch   (no loads, 4 KB written per frame)")
print(f"istft+phase    {kb:8.2f} us/iter     {F*20516/kb/1e3:8.1f} GB/s")
