"""Per-strip column layout of the structured-grid kernel's packed V: tried and not merged (r3_ab_grid2_column_map.txt).

  python profiles/tools/time_grid2_column_map.py --table        (CPU) tiles per (node row, strip) of the workloads' V
                                                                in the natural column order (what vo_grid2_kernel runs)
                                                                and after a per-strip first-fit column layout
  python profiles/tools/time_grid2_column_map.py [--iters N]    (GPU) torch.profiler device times of the packing kernel
                                                                and the residual kernel of the config-2 step's VO call
                                                                (pack_weights, then the prepacked residual); one JSON line
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)


def first_fit(row_masks, NT):
    """The layout rule: rows in order; a row whose columns sit in one tile takes the first such tile, else the
    first tile with room for its missing columns, else a new tile; None = natural layout (more than NT tiles, or a row
    with more than 8 columns)."""
    tiles, tile_of = [], []
    for rm in row_masks:
        if rm == 0:
            tile_of.append(None)
            continue
        hit = next((i for i, t in enumerate(tiles) if rm & ~t['set'] == 0), None)
        if hit is None:
            hit = next((i for i, t in enumerate(tiles) if bin(rm & ~t['set']).count('1') <= 8 - t['n']), None)
            if hit is None:
                if len(tiles) == NT or bin(rm).count('1') > 8:
                    return None
                tiles.append({'set': 0, 'n': 0})
                hit = len(tiles) - 1
            add = rm & ~tiles[hit]['set']
            tiles[hit]['set'] |= rm
            tiles[hit]['n'] += bin(add).count('1')
        tile_of.append(hit)
    return tiles, tile_of


def strip_masks(V, nx, ny, NT):
    """[strip][node row] set of the non-zero main columns (< 8 NT) of V [d, m] on an nx x ny pixel grid."""
    ncol = nx - 1
    Vr = (V.reshape(ny + 1, ncol, V.shape[1])[:, :, :8 * NT] != 0)
    out = []
    for q in range(nx // 16):
        blk = Vr[:, 16 * q:16 * q + 16, :].any(axis=1)
        out.append([int(sum(1 << j for j in np.nonzero(blk[t])[0])) for t in range(ny + 1)])
    return out


def table(V, nx, ny, m):
    NT = m // 8 if (m % 8) <= 1 and m >= 8 else (m + 7) // 8
    masks = strip_masks(V, nx, ny, NT)
    natural = compact = rows = 0
    per_strip, dfma = [], 0
    for q, rms in enumerate(masks):
        res = first_fit(rms, NT)
        for rm in rms:
            if rm:
                rows += 1
                natural += sum(1 for tt in range(NT) if (rm >> (8 * tt)) & 0xff)
        if res is None:
            per_strip.append("natural")
            compact += sum(sum(1 for tt in range(NT) if (rm >> (8 * tt)) & 0xff) for rm in rms if rm)
        else:
            tiles, tile_of = res
            per_strip.append(len(tiles))
            compact += sum(1 for t in tile_of if t is not None)
    if NT * 8 < m:
        Vx = V.reshape(ny + 1, nx - 1, m)[:, :, 8 * NT]
        dfma = sum(bool((Vx[:, 16 * q:16 * q + 16] != 0)[t].any()) for q in range(nx // 16) for t in range(ny + 1))
    return {"nx": nx, "m": m, "NT": NT, "tiles_per_row_strip_natural": natural / rows,
            "tiles_per_row_strip_column_map": compact / rows, "tiles_per_strip": per_strip,
            "rows_with_dfma_column": dfma / ((ny + 1) * (nx // 16)) if dfma else 0.0}


def cpu_table():
    from gpde_b200.workloads import Workload
    out = {}
    for name in ("cfg2", "cfg1"):
        w = Workload(name, B=8, seed=0)
        nx = w.physics["fom"].mesh.nx
        out[name] = table(np.asarray(w.V), nx, nx, w.m)
        rng = np.random.RandomState(0)
        out[name + "_dense_gaussian"] = table(rng.normal(size=np.asarray(w.V).shape), nx, nx, w.m)
    for k, v in out.items():
        print(k, json.dumps(v))


def gpu_times(iters):
    import torch
    from gpde_b200.VirtualObservables import VoPlan
    from gpde_b200.workloads import Workload
    dev = torch.device("cuda", 0)
    w = Workload("cfg2", B=4096, seed=0)
    plan = VoPlan.cached(w.physics["fom"], dev, pixel_input=True)
    a, y, g, V = (torch.tensor(t, device=dev) for t in (np.exp(w.log_image), w.y, w.g_fom, w.V))
    pw = plan.pack_weights(V, w.B)

    def call():
        p = plan.pack_weights(V, w.B, out=pw)
        return plan.residual(a, y, g, p, a_is_log=False, sm_reserve=20)
    for _ in range(20):
        call()
    torch.cuda.synchronize(dev)
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            call()
        torch.cuda.synchronize(dev)
    times = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" and "vo_grid2" in e.name:
            key = "pack" if "pack" in e.name else "residual"
            times.setdefault(key, []).append(e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total)
    props = torch.cuda.get_device_properties(dev)
    rec = {"gpu": props.name, "iters": iters, "m": w.m, "B": w.B}
    for k, v in times.items():
        rec["us_" + k + "_median"] = float(np.median(v))
        rec["us_" + k + "_min"] = float(np.min(v))
        rec["n_" + k] = len(v)
    print(json.dumps(rec))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--table", action="store_true")
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    if args.table:
        cpu_table()
    else:
        gpu_times(args.iters)
