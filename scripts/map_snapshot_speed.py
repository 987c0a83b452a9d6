"""Time of map snapshots (svnicp_map_export / svnicp_map_import) against GetMap() on the same map.

python scripts/map_snapshot_speed.py [--calls N] [--json OUT]

Maps: "configs1", a saturated 1 m / 20-point local map built from 12 scans of the 64-beam synth drive (configs[1] size), and
"configs4", a 1 m / 20-point map of ~10.8 M points (16 M uniform points in a 120 x 120 x 38 m box around the origin, so nearly
every voxel holds its 20 points; configs[4] size).  Per case: CUDA events around the blocking call (the map runs on its own stream
and every call returns when its results are in place), median and min over the calls.  Cases: Export / Import with host arrays
(the copies included; Export allocates fresh arrays, and the raw ABI call into host arrays that were touched before shows the cost
of their first touch) and with device tensors (no host transfer); GetMap() to the device and to the host.  Also the snapshot's
bytes (16 V + 12 Npts), the pageable copy rates measured with torch on the same byte count, and the card name and power limit.
Needs the GPU: there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 0xC0FFEE


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def timed(fn, calls):
    import torch
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st = torch.cuda.current_stream()
    for _ in range(2):
        fn()
    ts = []
    for _ in range(calls):
        ev0.record(st)
        fn()
        ev1.record(st)
        ev1.synchronize()
        ts.append(ev0.elapsed_time(ev1))
    return float(np.median(ts)), float(np.min(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    import svn_icp_b200 as sv
    from svn_icp_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("map_snapshot_speed: no CUDA device (this measurement has no CPU fallback)")
    name, limit = card()
    print(f"card: {name}; power limit, max SM clock: {limit}", flush=True)
    res = dict(card=name, power_limit_and_max_clock=limit, maps=[])

    def configs1():
        m = sv.VoxelHashMap(1.0, 100.0, 20)
        world = synth.make_world(SEED)
        for k in range(12):
            pts, (R, t) = synth.make_scan(world, k, "64", SEED)
            m.AddPointCloud(pts.astype(np.float32), R, t)
        return m

    def configs4():
        m = sv.VoxelHashMap(1.0, 1e4, 20, capacity_voxels=1 << 20)
        pts = np.random.default_rng(4).uniform([-60, -60, -19], [60, 60, 19], (16_000_000, 3)).astype(np.float32)
        m.AddPointCloud(pts, np.eye(3), np.zeros(3))
        return m

    for label, make in (("configs1", configs1), ("configs4", configs4)):
        m = make()
        V, N = m.Size(), m.PointCount()
        snap_bytes = 16 * V + 12 * N
        print(f"{label}: {V} voxels, {N} points ({N / V:.1f} per voxel), snapshot {snap_bytes / 1e6:.1f} MB", flush=True)
        s = m.Export()
        vox = torch.zeros((V, 3), dtype=torch.int32, device="cuda")
        cnt = torch.zeros(V, dtype=torch.int32, device="cuda")
        xyz = torch.zeros((N, 3), dtype=torch.float32, device="cuda")
        b = sv.VoxelHashMap(m.voxel_size_, m.max_range_, m.max_pointscount_, capacity_voxels=max(V, 1 << 19))
        dev = torch.empty(snap_bytes, dtype=torch.uint8, device="cuda")
        host = torch.empty(snap_bytes, dtype=torch.uint8)
        hv, hc, hx = np.ones((V, 3), np.int32), np.ones(V, np.int32), np.ones((N, 3), np.float32)  # host arrays touched once
        raw = lambda: m._check(m._lib.svnicp_map_export(m._m, sv._p(hv), sv._p(hc), sv._p(hx), V, N, 0), "Export")  # noqa: E731
        cases = [("export_host", m.Export),
                 ("export_host_reused_arrays", raw),
                 ("export_device", lambda: m.ExportDevice(vox.data_ptr(), cnt.data_ptr(), xyz.data_ptr())),
                 ("import_host", lambda: b.Import(s)),
                 ("import_device", lambda: b.ImportDevice(vox.data_ptr(), cnt.data_ptr(), xyz.data_ptr(), V, N)),
                 ("getmap_device", lambda: m.GetMapDevice()),
                 ("getmap_host", lambda: m.GetMap()),
                 ("copy_d2h_pageable", lambda: host.copy_(dev)),
                 ("copy_h2d_pageable", lambda: dev.copy_(host))]
        row = dict(map=label, voxels=V, points=N, snapshot_bytes=snap_bytes, getmap_bytes_host=24 * N, cases={})
        for cname, fn in cases:
            med, mn = timed(fn, args.calls)
            row["cases"][cname] = dict(ms_median=med, ms_min=mn)
            print(f"{label} {cname:18s}: {med:8.3f} ms median, {mn:8.3f} ms min", flush=True)
        b.Import(s)
        assert b.Export().points.tobytes() == s.points.tobytes()
        for d in ("d2h", "h2d"):
            row[f"copy_{d}_GBps"] = snap_bytes / (row["cases"][f"copy_{d}_pageable"]["ms_median"] * 1e6)
        print(f"{label}: pageable copy rate at the snapshot's size: D2H {row['copy_d2h_GBps']:.1f} GB/s, "
              f"H2D {row['copy_h2d_GBps']:.1f} GB/s", flush=True)
        res["maps"].append(row)
        del m, b
    print(json.dumps(res))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
