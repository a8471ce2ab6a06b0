"""Per-CTA %globaltimer timeline of two consecutive K1 launches (debug build with -DMG_TIMELINE, see
mg_step.cu): where a step's fixed cost goes (launch gap, prologue, dependency wait, first tile, drain).
usage: MINIGRID_B200_LIB=.../libminigrid_b200_tl.so python scripts/timeline.py [n_envs ...]"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from minigrid_b200 import MinigridVecEnv, _lib

sizes = [int(s) for s in sys.argv[1:]] or [4736, 262144]
L = _lib.load()
raw = ctypes.CDLL(os.environ["MINIGRID_B200_LIB"])
for n in sizes:
    e = MinigridVecEnv("MiniGrid-DoorKey-8x8-v0", n); e.reset(seed=0)
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
    rc = raw.mg_debug_timeline(ctypes.c_void_p(buf.ctypes.data), 0)  # DoorKey-8x8: tiled layout
    assert rc == 0, rc
    ncta = int((buf[0, :, 0] != 0).sum())
    tl = buf[:, :ncta, :].astype(np.int64)
    # order the two slots in time
    a, b = (0, 1) if tl[0, :, 0].min() < tl[1, :, 0].min() else (1, 0)
    t0 = tl[a, :, 0].min()
    def stat(x): return f"min {x.min()/1e3:7.2f}  med {np.median(x)/1e3:7.2f}  max {x.max()/1e3:7.2f}"
    names = ["entry", "prologue done", "after griddep wait", "first tile arrived (warp0)", "first tile done (warp0)",
             "warp0 exit", "last warp exit", "first warp exit"]
    print(f"== n={n}  (us relative to the first CTA entry of launch A; B is the next launch)")
    for tag, k in (("A", a), ("B", b)):
        for i, nm in enumerate(names):
            print(f"  {tag} {nm:28s} {stat(tl[k, :, i] - t0)}")
    print(f"  period (B entry min - A entry min): {(tl[b,:,0].min() - tl[a,:,0].min())/1e3:.2f} us;  "
          f"A last exit -> B first 'after wait': {(tl[b,:,2].min() - tl[a,:,6].max())/1e3:.2f} us")
    if os.environ.get("TIMELINE_DUMP"):
        np.save(os.environ["TIMELINE_DUMP"] + f"_{n}.npy", np.stack([tl[a] - t0, tl[b] - t0]))
    res = np.unique(np.diff(np.sort(tl[a].ravel())))
    print("  timer granularity (smallest nonzero delta, ns):", res[res > 0][:3])
    del e, g
