"""One Griffin-Lim call on the cfg3 shape (or B T n_iter from argv) -- the command ncu captures for profiles/."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import spev_tts_b200 as sp
dev = torch.device("cuda", 0)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
T = int(sys.argv[2]) if len(sys.argv) > 2 else 800
n_iter = int(sys.argv[3]) if len(sys.argv) > 3 else 6
ctx = sp.Context.get(dev, fmin=0.0, fmax=8000.0)
fb = sp.make_batch(ctx, n_frames=[T] * B, with_chunks=True)
g = torch.Generator(device=dev).manual_seed(0)
S = torch.rand(fb.n_frames, 520, generator=g, device=dev)
for _ in range(2):
    y = sp.griffinlim_flat(S, fb, ctx, n_iter=n_iter, seed=7)
torch.cuda.synchronize()
print("ok", float(y.abs().mean()))
