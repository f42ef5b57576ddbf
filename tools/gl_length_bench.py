"""Time spev_griffinlim with and without an explicit output length (librosa's ``length=``) at cfg3.

    python tools/gl_length_bench.py [--parent-lib PATH] [--rounds 6] [--calls 10] [--out DIR]

cfg3 is 16 items x 800 frames, 60 iterations, with seeded magnitudes and initial phases.  Each round times --calls
back-to-back calls with device events, once per variant, the variants alternating round by round:
  default  : no length, this build ((T-1)*256 = 204,544 samples per item)
  length   : length = 204,799 per item (T*256 - 1: the worst case, a 255-sample tail re-analysed every iteration)
  parent   : no length, another build of the library (--parent-lib, e.g. the parent commit's), for outputs and time,
             on tile tables planned by that build's own planners.
The default output must be bit-identical to the parent's.  The card name and power limit are printed with the numbers.
Prints one JSON line; --out also writes it to DIR/gl_length_bench.json.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import spev_tts_b200 as sp  # noqa: E402
from spev_tts_b200 import _lib  # noqa: E402

B, T, N_ITER = 16, 800, 60
L = T * 256 - 1


class Lib:
    """One build of the library: its ctx and a spev_griffinlim call."""

    def __init__(self, path, dev):
        if path is None:
            self.lib = _lib.load()
        else:
            self.lib = C.CDLL(os.path.abspath(path))
            for name in ("spev_abi_version", "spev_create", "spev_destroy", "spev_griffinlim",
                         "spev_griffinlim_workspace_bytes", "spev_last_error", "spev_plan_frame_tiles", "spev_plan_chunk_tiles"):
                res, args = _lib._SIGS[name]
                getattr(self.lib, name).restype = res
                getattr(self.lib, name).argtypes = args
        h = C.c_void_p()
        self._check(self.lib.spev_create(C.byref(h), dev.index, 22050, 1024, 256, 1024, 80, 0.0, 8000.0))
        self.handle = h

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(f"spev call failed ({rc}): {self.lib.spev_last_error().decode(errors='replace')}")

    def replan(self, fb, dev):
        """The batch ``fb`` with tile tables from this build's own planners.  Builds before ABI 3 plan the default
        output layout from NULL layout arrays (chunk tiles with lo = hi = 0)."""
        layout = [fb.out_off, fb.out_len] if self.lib.spev_abi_version() >= 3 else [None, None]
        args = [fb.frames.ctypes.data] + [None if a is None else a.ctypes.data for a in layout] + [fb.n_items]
        tables = []
        for fn in (self.lib.spev_plan_frame_tiles, self.lib.spev_plan_chunk_tiles):
            n = fn(*args, None)
            if n < 0:
                self._check(n)
            tables.append(np.empty(n, dtype=sp.batch.TILE_DTYPE))
            fn(*args, tables[-1].ctypes.data)
        ft, ct = tables
        table = torch.from_numpy(np.concatenate([ft.view(np.uint8), ct.view(np.uint8), fb.frame_off.view(np.uint8)])).to(dev)
        d = _lib.SpevBatch()
        d.n_items, d.n_frames, d.n_ftiles, d.n_ctiles = fb.n_items, fb.n_frames, len(ft), len(ct)
        d.ftiles, d.ctiles, d.frame_off = table.data_ptr(), table.data_ptr() + ft.nbytes, table.data_ptr() + ft.nbytes + ct.nbytes
        return types.SimpleNamespace(desc=d, table=table, n_out_samples=fb.n_out_samples)

    def griffinlim(self, fb, S, ph, y, ws, st):
        self._check(self.lib.spev_griffinlim(self.handle, fb.desc, S.data_ptr(), S.shape[1], ph.data_ptr(), 7, N_ITER, 0.99,
                                             y.data_ptr(), ws.data_ptr(), ws.numel(), st))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gl_length_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    ctx = sp.Context.get(dev, fmin=0.0, fmax=8000.0)
    fb_def = sp.make_batch(ctx, n_frames=[T] * B, with_chunks=True)
    fb_len = sp.make_batch(ctx, n_frames=[T] * B, with_chunks=True, out_len=[L] * B)
    g = torch.Generator(device=dev).manual_seed(3)
    S = torch.rand(B * T, _lib.SPEC_LD, generator=g, device=dev)
    ph = torch.rand(B * T, 513, generator=g, device=dev) * 6.2831853
    ws = torch.empty(ctx.lib.spev_griffinlim_workspace_bytes(B * T), dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    cur = Lib(None, dev)
    libs = {"default": (cur, fb_def), "length": (cur, fb_len)}
    if a.parent_lib:
        parent = Lib(a.parent_lib, dev)
        libs["parent"] = (parent, parent.replan(fb_def, dev))
    ys = {k: torch.empty(fb.n_out_samples, device=dev) for k, (_, fb) in libs.items()}

    def run(k, n):
        lib, fb = libs[k]
        for _ in range(n):
            lib.griffinlim(fb, S, ph, ys[k], ws, st)

    for k in libs:                                       # warm-up: module load, first launches
        run(k, 2)
    torch.cuda.synchronize(dev)
    times = {k: [] for k in libs}
    order = list(libs)
    for r in range(a.rounds):
        for k in (order if r % 2 == 0 else order[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            run(k, a.calls)
            e1.record()
            torch.cuda.synchronize(dev)
            times[k].append(e0.elapsed_time(e1) / a.calls)
    res = {"shape": f"{B} x {T} frames, {N_ITER} iterations", "length": L, "calls_per_round": a.calls,
           "gpu": torch.cuda.get_device_name(dev)}
    try:
        res["power_limit_w"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        res["power_limit_w"] = f"unavailable ({e})"
    for k, v in times.items():
        res[f"{k}_ms"] = {"min": round(min(v), 4), "max": round(max(v), 4), "median": round(float(np.median(v)), 4)}
    if "parent" in libs:
        res["default_bit_identical_to_parent"] = bool(torch.equal(ys["default"], ys["parent"]))
    off = fb_len.out_sample_off()
    yl = ys["length"]
    res["length_finite"] = bool(torch.isfinite(torch.cat([yl[off[i]: off[i] + L] for i in range(B)])).all())
    res["length_over_default"] = round(float(np.median(times["length"]) / np.median(times["default"])), 4)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "gl_length_bench.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
