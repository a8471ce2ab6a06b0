"""Per-CTA timeline of one K1 launch with DESYNCHRONISED episodes (debug build with -DMG_TIMELINE): how long a tile that
regenerates environments takes, when the last of them finishes, and whether it is what a CTA ends on.
usage: MINIGRID_B200_LIB=.../libminigrid_b200_tl.so python scripts/timeline2.py [env_id] [n_envs]"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from minigrid_b200 import MinigridVecEnv, _lib

env_id = sys.argv[1] if len(sys.argv) > 1 else "MiniGrid-DoorKey-8x8-v0"
n = int(sys.argv[2]) if len(sys.argv) > 2 else 262144
L = _lib.load()
raw = ctypes.CDLL(os.environ["MINIGRID_B200_LIB"])
for desync in (False, True):
    e = MinigridVecEnv(env_id, n); e.reset(seed=0)
    if desync:
        st = e.get_state()
        st["agent"][:, 5] = torch.randint(0, e.max_steps, (n,), device="cuda", dtype=torch.int32)
        e.set_state(agent=st["agent"])
    acts = torch.randint(0, 7, (64, n), device="cuda", dtype=torch.int32)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for t in range(20): e.step(acts[t % 64])
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for t in range(64): e.step(acts[t])
    for _ in range(5): g.replay()
    torch.cuda.synchronize()
    buf = np.zeros((2, 160, 16), np.uint64)
    layout = int(os.environ.get("TL_LAYOUT", "0"))  # the env's layout: 0 tiled, 1 window
    assert raw.mg_debug_timeline(ctypes.c_void_p(buf.ctypes.data), layout) == 0
    ncta = int((buf[0, :, 0] != 0).sum())
    tl = buf[:, :ncta, :].astype(np.int64)
    a, b = (0, 1) if tl[0, :, 0].min() < tl[1, :, 0].min() else (1, 0)
    A = tl[a]
    t0 = A[:, 2].min()  # release of griddepcontrol.wait
    us = lambda x: x / 1e3
    print(f"== {env_id} n={n} desync={desync}: {ncta} CTAs; period {us(tl[b,:,0].min() - tl[a,:,0].min()):.2f} us")
    B = tl[b]
    for nm, k in (("entry", 0), ("prologue done", 1), ("wait released", 2), ("warp0 first tile in", 3), ("warp0 exit", 5), ("last warp exit", 6)):
        print(f"   A {nm:22s} min {us(A[:,k].min()-t0):7.2f} med {us(np.median(A[:,k])-t0):7.2f} max {us(A[:,k].max()-t0):7.2f}   |  B min {us(B[:,k].min()-t0):7.2f} med {us(np.median(B[:,k])-t0):7.2f} max {us(B[:,k].max()-t0):7.2f}")
    print(f"   last warp exit (rel. to wait release): min {us(A[:,6].min()-t0):.2f} med {us(np.median(A[:,6])-t0):.2f} max {us(A[:,6].max()-t0):.2f}")
    print(f"   order list ready: med {us(np.median(A[:,13][A[:,13]>0]) - t0) if (A[:,13]>0).any() else -1:.2f}")
    hot = A[:, 8]
    print(f"   regenerating tiles per CTA: mean {hot.mean():.2f} max {hot.max()}; longest regenerating tile: med {us(np.median(A[:,9][hot>0])) if (hot>0).any() else 0:.2f} max {us(A[:,9].max()):.2f} us; longest plain tile: med {us(np.median(A[:,10])):.2f} max {us(A[:,10].max()):.2f}")
    if (hot > 0).any():
        m = hot > 0
        print(f"   end of the last regenerating tile (rel.): med {us(np.median(A[m,11]) - t0):.2f} max {us(A[m,11].max()-t0):.2f}; its CTA's exit - that: med {us(np.median(A[m,6]-A[m,11])):.2f} min {us((A[m,6]-A[m,11]).min()):.2f}; largest pull index of a regenerating tile: med {np.median(A[m,12]):.0f} max {A[m,12].max()}")
        order = np.argsort(A[:, 6])[-8:]
        for c in order:
            print(f"     slow CTA {c}: exit {us(A[c,6]-t0):.2f}  regen tiles {A[c,8]}  longest regen {us(A[c,9]):.2f}  last regen end {us(A[c,11]-t0) if A[c,8] else 0:.2f}  longest plain {us(A[c,10]):.2f}")
    del e, g
