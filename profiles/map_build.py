"""Corrected global map on one GPU: build time, throughput, oracle parity, and the 8-bit vs 11-bit sort digits.

    python profiles/map_build.py --out map_build.json

Builds the maps of the first 600 and of all 2761 keyframes of synth.make_sequence(5, 2761, pts_per_keyframe=30000) (the
KITTI-05-shaped sequence of bench.py's sequence workload) at 0.3 m (a 24-bit grid: 8-bit sort digits) and 0.1 m (28 bits:
11-bit digits).  Each map is built --warmup times, then timed --reps times with a host clock around the build and a
synchronise of the context; the median is reported, with points/s and algorithmic bytes/s (128 B per merged point: 16 + 16
transform, 16 + 8 keys, 3 x 16 sort passes, 4 run heads, 20 centroids).  Every map is compared bit for bit with the CPU
oracle (transform_pcd + voxelize, one thread), which is timed on the same input.

The sort-digit comparison builds the library a second time with -DB200REG_NO_SORT8 (into a temporary directory) and times
the 0.3 m map of all keyframes with both libraries, alternating them, in the same process.  The GPU's name and power limit
are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "fast-lio-sam-qn_b200"))

BYTES_PER_POINT = 128


def build_variant(out_dir, defines):
    """The library with extra -D flags, compiled into out_dir (the tree is not touched)."""
    from b200reg import build as B
    def cc(src):
        obj = os.path.join(out_dir, src.replace(".cu", ".o"))
        cmd = [B.NVCC] + B.FLAGS + B.EXTRA.get(src, []) + ["-D" + d for d in defines] + ["-c", os.path.join(B.CSRC, src), "-o", obj]
        subprocess.run(cmd, check=True, capture_output=True)
        return obj
    with ThreadPoolExecutor(len(B.SOURCES)) as ex:
        objs = list(ex.map(cc, B.SOURCES))
    lib = os.path.join(out_dir, "libb200reg.so")
    subprocess.run([B.NVCC, "-shared", "-o", lib, "-ccbin", "/usr/bin/g++"] + objs + ["-ldl", "-lpthread"], check=True, capture_output=True)
    return lib


class Engine:
    """A context and a keyframe store on one build of libb200reg.so (plain ctypes: two builds can live in one process)."""

    def __init__(self, path, seq, n_points):
        self.l = C.CDLL(path)
        self.l.b200reg_last_error.restype = C.c_char_p
        self.l.b200reg_map_size.restype = C.c_size_t
        self.ctx, self.kf = C.c_void_p(), C.c_void_p()
        self._ok(self.l.b200reg_ctx_create(0, C.byref(self.ctx)))
        self._ok(self.l.b200reg_keyframes_create(self.ctx, C.byref(self.kf)))
        self._ok(self.l.b200reg_keyframes_reserve(self.ctx, self.kf, C.c_size_t(n_points)))
        for c, T, t in zip(seq["clouds"], seq["poses"], seq["stamps"]):
            a = np.ascontiguousarray(c[:, :4], np.float32)
            P = np.ascontiguousarray(T, np.float64).reshape(16)
            rc = self.l.b200reg_keyframes_add(self.ctx, self.kf, a.ctypes.data_as(C.c_void_p), C.c_size_t(len(a)), C.c_size_t(16),
                                              P.ctypes.data_as(C.c_void_p), C.c_double(t))
            if rc < 0:
                self._ok(rc)
        self._ok(self.l.b200reg_ctx_synchronize(self.ctx))

    def _ok(self, rc):
        if rc != 0:
            raise RuntimeError("b200reg error %d: %s" % (rc, self.l.b200reg_last_error().decode()))

    def build(self, n_keyframes, leaf, fetch=False):
        """-> (seconds for build + synchronise, records or None, voxelized)"""
        h = C.c_void_p()
        t0 = time.perf_counter()
        self._ok(self.l.b200reg_map_build(self.ctx, self.kf, int(n_keyframes), C.c_double(leaf), C.byref(h)))
        self._ok(self.l.b200reg_ctx_synchronize(self.ctx))
        dt = time.perf_counter() - t0
        out = None
        if fetch:
            out = np.empty((int(self.l.b200reg_map_size(h)), 4), np.float32)
            self._ok(self.l.b200reg_map_get(self.ctx, h, out.ctypes.data_as(C.c_void_p)))
        vox = bool(self.l.b200reg_map_voxelized(h))
        self._ok(self.l.b200reg_map_destroy(self.ctx, h))
        return dt, out, vox

    def close(self):
        self.l.b200reg_keyframes_destroy(self.ctx, self.kf)
        self.l.b200reg_ctx_destroy(self.ctx)


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: no GPU to measure on")
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--keyframes", default="600,2761")
    ap.add_argument("--leaves", default="0.3,0.1")
    ap.add_argument("--pts", type=int, default=30000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--threads", type=int, default=8, help="threads of the synthetic-sequence generator")
    ap.add_argument("--no-variant", action="store_true", help="skip the build without 8-bit sort digits")
    args = ap.parse_args()
    kfs = [int(k) for k in args.keyframes.split(",")]
    leaves = [float(x) for x in args.leaves.split(",")]
    res = dict(gpu=gpu_info(), sequence="synth.make_sequence(5, %d, pts_per_keyframe=%d)" % (max(kfs), args.pts),
               reps=args.reps, warmup=args.warmup, bytes_per_point=BYTES_PER_POINT, maps=[])
    from b200reg import synth
    from b200reg.build import build_native
    from oracle import oracle as orc
    t = time.perf_counter()
    seq = synth.make_sequence(5, max(kfs), pts_per_keyframe=args.pts, threads=args.threads)
    res["synth_s"] = round(time.perf_counter() - t, 1)
    n_points = sum(len(c) for c in seq["clouds"])
    main_lib = build_native()
    eng = Engine(main_lib, seq, n_points)
    for nk in kfs:
        t = time.perf_counter()
        merged = np.concatenate([orc.transform_pcd(seq["clouds"][i], seq["poses"][i]) for i in range(nk)])
        oracle_transform_s = time.perf_counter() - t
        for leaf in leaves:
            for _ in range(args.warmup):
                eng.build(nk, leaf)
            times = [eng.build(nk, leaf)[0] for _ in range(args.reps)]
            _, got, vox = eng.build(nk, leaf, fetch=True)
            t = time.perf_counter()
            want = orc.voxelize(merged, leaf)
            oracle_voxelize_s = time.perf_counter() - t
            ms = float(np.median(times)) * 1e3
            n = len(merged)
            row = dict(keyframes=nk, leaf=leaf, points=n, voxels=len(got), voxelized=vox, median_ms=round(ms, 3),
                       min_ms=round(min(times) * 1e3, 3), max_ms=round(max(times) * 1e3, 3),
                       points_per_s=round(n / (ms * 1e-3)), algo_gb_per_s=round(BYTES_PER_POINT * n / (ms * 1e-3) / 1e9, 1),
                       oracle_s=round(oracle_transform_s + oracle_voxelize_s, 2),
                       oracle_transform_s=round(oracle_transform_s, 2), oracle_voxelize_s=round(oracle_voxelize_s, 2),
                       bit_exact=bool(np.array_equal(got, want)))
            print(json.dumps(row), flush=True)
            res["maps"].append(row)
        del merged
    if not args.no_variant:
        nk, leaf = max(kfs), 0.3
        with tempfile.TemporaryDirectory() as d:
            alt = Engine(build_variant(d, ["B200REG_NO_SORT8"]), seq, n_points)
            for _ in range(args.warmup):
                eng.build(nk, leaf)
                alt.build(nk, leaf)
            t8, t11 = [], []
            for _ in range(args.reps):
                t8.append(eng.build(nk, leaf)[0])
                t11.append(alt.build(nk, leaf)[0])
            _, a, _ = eng.build(nk, leaf, fetch=True)
            _, b, _ = alt.build(nk, leaf, fetch=True)
            alt.close()
        res["sort_digits"] = dict(keyframes=nk, leaf=leaf, median_ms_8bit=round(float(np.median(t8)) * 1e3, 3),
                                  median_ms_11bit=round(float(np.median(t11)) * 1e3, 3), same_records=bool(np.array_equal(a, b)),
                                  note="same process, alternating; 11-bit = the library built with -DB200REG_NO_SORT8")
        print(json.dumps(res["sort_digits"]), flush=True)
    eng.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    if not all(r["bit_exact"] for r in res["maps"]):
        sys.exit("map differs from the oracle")


if __name__ == "__main__":
    main()
