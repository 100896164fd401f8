"""A/B of two builds of libpom_b200.so on one GPU: the record array in compressible device memory (this build) against
cudaMalloc (a build that predates it).  Prints one JSON line with the card and what the driver reports, then one line per
leg with every round's figure for both builds, their medians and spreads.

    python tools/bench_compressible.py --base PATH/libpom_b200.so [--this PATH/libpom_b200.so] [--rounds R] [--steps K]

--this defaults to the tree's own build.

Each round runs both builds, one after the other in a process of its own (POM_B200_LIB selects the library), and the
order swaps from round to round, so that other load on the machine falls on both alike.  The legs are bench.py's:
  tick      the timed region: 1 Mi envs, AUTORESET | COUNT | POM_STEP_OVERLAP, moves from a ring of 256 move sets on the
            device, K ticks after the 96-tick preroll and 20 warm-up ticks
  single    one launch per tick over the whole batch, ticks strictly one after the other (roofline.single_launch)
  strong2   the tick loop on 0.5 Mi envs: one GPU's share of legs.strong on two GPUs (the records partly fit the L2)
  big       the tick loop on 4 Mi envs (roofline.big_batch)
  rollout   legs.rollout: fused 800-tick rollout of 0.5 Mi envs
  expand    legs.expand: 4,096 roots x 1,296 children, clone + one Step each, 10 calls back to back
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THIS_LIB = os.path.join(ROOT, "pomcpp_b200", "libpom_b200.so")

SEED = 20240229
N = 1 << 20
RING = 256
PREROLL = 96


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in out.stdout.strip().split(",")])) if out.returncode == 0 else {}


class AllocProp(C.Structure):
    """CUmemAllocationProp (cuda.h)"""
    _fields_ = [("type", C.c_int), ("requestedHandleTypes", C.c_int), ("loc_type", C.c_int), ("loc_id", C.c_int),
                ("win32HandleMetaData", C.c_void_p), ("compressionType", C.c_ubyte), ("gpuDirectRDMACapable", C.c_ubyte),
                ("usage", C.c_ushort), ("reserved", C.c_ubyte * 4)]


def driver_info(device=0):
    """what the driver says about generic compression on `device`: the attribute and the compressible granularity"""
    cu = C.CDLL("libcuda.so.1")
    dev, v = C.c_int(), C.c_int()
    out = {}
    if cu.cuInit(0) != 0 or cu.cuDeviceGet(C.byref(dev), device) != 0:
        return {"error": "cuInit / cuDeviceGet failed"}
    for name, attr in (("generic_compression_supported", 107), ("virtual_memory_management_supported", 102)):
        out[name] = v.value if cu.cuDeviceGetAttribute(C.byref(v), attr, dev) == 0 else None
    p = AllocProp(type=1, loc_type=1, loc_id=dev.value, compressionType=1)
    g = C.c_size_t()
    for name, which in (("granularity_minimum", 0), ("granularity_recommended", 1)):
        out[name] = g.value if cu.cuMemGetAllocationGranularity(C.byref(g), C.byref(p), which) == 0 else None
    return out


def tick_loop(pb, b, moves, n_ring_envs, steps, flags, warm):
    for w in range(warm):
        b.step(moves.value + 4 * n_ring_envs * (w % RING), flags)
    b.sync()
    b.clear_stats()
    b.event(0)
    for k in range(steps):
        b.step(moves.value + 4 * n_ring_envs * ((warm + k) % RING), flags)
    b.event(1)
    ms = b.elapsed_ms() / steps
    assert b.stats().env_steps == b.n * steps
    return ms


def child(steps):
    sys.path.insert(0, ROOT)
    import numpy as np
    import pomcpp_b200 as pb
    pb.bind_thread_near(0)
    plain = pb.STEP_AUTORESET | pb.STEP_COUNT
    over = plain | pb.STEP_OVERLAP
    res = {}

    def compressed(x):
        try:
            return x.records_compressed()
        except AttributeError:                              # a build that predates the query
            return None

    b = pb.Batch(N, n_templates=4096, max_ticks=800)
    res["records_compressed"] = compressed(b)
    moves = b.alloc(4 * N * RING)
    for t in range(RING):
        b.generate_moves(moves.value + 4 * N * t, SEED, 100000 + t, 6)
    b.rollout(PREROLL, SEED, 0, 0)
    res["single_ms"] = tick_loop(pb, b, moves, N, min(200, steps), plain, 5)
    res["tick_ms"] = tick_loop(pb, b, moves, N, steps, over, 20)

    e = pb.Batch(4096 * 1296, n_templates=16, empty=True)
    roots = (np.arange(4096, dtype=np.uint32) * 251) % N
    e.expand_step_from(b, roots, 1296, 0)
    e.sync()
    e.event(0)
    for _ in range(10):
        e.expand_step_from(b, roots, 1296, 0)
    e.event(1)
    res["expand_ms"] = e.elapsed_ms() / 10
    e.close()

    s = pb.Batch(N // 2, n_templates=4096, max_ticks=800)
    s.rollout(PREROLL, SEED, 0, 0)
    res["strong2_ms"] = tick_loop(pb, s, moves, N, steps, over, 5)
    s.close()

    r = pb.Batch(N // 2, n_templates=4096, max_ticks=800)
    r.rollout(64, SEED, 0, 0)
    r.sync()
    r.event(0)
    r.rollout(800, SEED, 64, 0)
    r.event(1)
    res["rollout_ms"] = r.elapsed_ms()
    r.close()
    b.free(moves)
    b.close()

    big = 4 * N
    g = pb.Batch(big, n_templates=4096, max_ticks=800)
    res["big_records_compressed"] = compressed(g)
    g.rollout(PREROLL, SEED, 0, 0)
    gm = g.alloc(4 * big * 6)
    for t in range(6):
        g.generate_moves(gm.value + 4 * big * t, SEED, 200000 + t, 6)
    g.sync()
    for w in range(4):
        g.step(gm.value + 4 * big * (w % 6), over)
    g.sync()
    g.event(0)
    for k in range(20):
        g.step(gm.value + 4 * big * (k % 6), over)
    g.event(1)
    res["big_ms"] = g.elapsed_ms() / 20
    g.free(gm)
    g.close()
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", help="the library to compare against (a build that allocates its records with cudaMalloc)")
    ap.add_argument("--this", default=THIS_LIB, help="the build under test")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a.steps)
        return
    if not a.base:
        ap.error("--base is required")
    libs = {"base": os.path.abspath(a.base), "this": os.path.abspath(a.this)}
    print(json.dumps({"gpu": gpu_info(), "driver": driver_info(), "steps": a.steps, "rounds": a.rounds,
                      **{k: os.path.relpath(v, ROOT) for k, v in libs.items()}}), flush=True)
    runs = {k: [] for k in libs}
    for r in range(a.rounds):
        for k in (("base", "this") if r % 2 == 0 else ("this", "base")):
            env = dict(os.environ, POM_B200_LIB=libs[k])
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", "--steps", str(a.steps)],
                                 env=env, capture_output=True, text=True)
            if out.returncode != 0:
                sys.exit("%s build, round %d failed:\n%s%s" % (k, r, out.stdout, out.stderr))
            runs[k].append(json.loads(out.stdout.strip().splitlines()[-1]))
    print(json.dumps({"records_compressed": {k: [x["records_compressed"] for x in runs[k]] for k in libs},
                      "big_records_compressed": {k: [x["big_records_compressed"] for x in runs[k]] for k in libs}}), flush=True)
    for leg in ("tick", "single", "strong2", "big", "rollout", "expand"):
        line = {"leg": leg, "unit": "ms"}
        for k in libs:
            v = [x[leg + "_ms"] for x in runs[k]]
            s = sorted(v)
            line[k] = {"median": s[len(s) // 2], "spread": (s[-1] - s[0]) / s[len(s) // 2], "rounds": v}
        line["this_over_base"] = line["this"]["median"] / line["base"]["median"]
        line["gpu"] = gpu_info()
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
