"""Tuning aid: per-phase clocks of lv_ieskf_step_kernel (library built with EXTRA=-DLV_STEP_TIMING)."""
import ctypes, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as G, bench
lv = G.load_package()
prm = lv.params_from_yaml(lv.CONFIG_DIR + "/xaloc.yaml", max_map_points=bench.MAP_POINTS + 4 * 65536, max_points=65536)
world, mp, sweeps, x_props, truths = bench.make_scene(lv, 0, n_sweeps=2, prm=prm)
x0, P0 = lv.init_state_host(prm)
loc = lv.Localizer(prm); loc.map_build(mp)
buf = (ctypes.c_longlong * 64)()
rows = []
for it in range(12):
    loc.set_state(x_props[it % 2], P0)
    if it % 2: loc.flush_l2()
    loc.correct(sweeps[it % 2])
    loc.L.lv_debug_step_clocks(buf)
    c = np.array(buf[:10], dtype=np.int64)
    rows.append(np.diff(c))
    b = buf
    ph = [b[1] - b[0], b[2] - b[1], b[5] - b[3], b[6] - b[5], b[7] - b[6], b[8] - b[7], b[9] - b[8]]
    print(("flush " if it % 2 else "warm  ") + " ".join(f"{d:7d}" for d in ph), " total", b[9] - b[0], " non-final", b[8] - b[0],
          " T1 tasks (pose, extr, grav, lin+conv):", [b[32 + k] - b[24 + k] for k in range(4)],
          " FIT block 1 (cycles): wait", b[57] - b[56], "loads", b[58] - b[57], "fit+row", b[59] - b[58], "stage", b[60] - b[59], "reduce", b[61] - b[60], "store+ticket", b[62] - b[61], "group sum", b[63] - b[62], "|",
          " solve: entry->loop", b[48] - b[5], "loop", b[49] - b[48], "store", b[52] - b[49], "exit->CK6", b[6] - b[52], " degeneracy test", b[51] - b[50])
print("phases: load | reduce | assemble A | solve (+degeneracy test) | K,dxs | tail | exit-P")
