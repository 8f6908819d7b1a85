"""Every host-side record of the library's plans, for an exact comparison of two builds of the same ABI (no GPU):
workspace size, every field of every stage record, launch records at 148, 132 and 64 SMs, generator and flow
gradient layouts, Langevin launch counts, packed-weight indices of two small plans, and the return code and error
text of invalid configs (one bad field, and every pair of bad fields).

    LSNF_LIB=tools/_ab/liblsnf_old.so python tools/plan_records.py dump old.json
    python tools/plan_records.py dump new.json
    python tools/plan_records.py compare old.json new.json [summary.json]
"""
import ctypes as C
import hashlib
import itertools
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from lsnf_b200 import _cabi  # noqa: E402

SMS = (148, 132, 64)
ARCHS = {"svhn": (100, 64), "cifar10": (128, 128), "celeba_crop": (100, 128), "celeba_hq256": (100, 128)}


def flat(v):
    if isinstance(v, C.Structure):
        return [flat(getattr(v, f)) for f, _ in v._fields_]
    if isinstance(v, C.Array):
        return [flat(x) for x in v]
    return v


def config(**kw):
    base = dict(arch=0, batch=100, nz=100, ngf=64, nc=3, f_depth=5, f_width=64, f_permutation=2, f_coupling=1,
                leak=0.2, gemm_impl=0, bwd_passes=3, train=0)
    base.update(kw)
    return base


def configs():
    out = []
    bench_like = [dict(arch=_cabi.ARCH[a], nz=nz, ngf=ngf, batch=b, f_width=fw) for a, (nz, ngf) in ARCHS.items()
                  for b, fw in ((100, 64), (8, 128), (1250, 64))]
    for c, bwd, train, impl in itertools.product(bench_like, (1, 3), (0, 1), (0, 1)):
        out.append(config(**c, bwd_passes=bwd, train=train, gemm_impl=impl))
    for nz, b in itertools.product((4, 132, 192, 256), (1, 57, 130)):   # tests/test_gpu_latent_sizes.py
        for train in (0, 1):
            out.append(config(arch=0, nz=nz, ngf=64, batch=b, train=train, f_permutation=1 if nz == 256 else 2))
    for train in (0, 1):
        out.append(config(arch=1, nz=256, ngf=128, batch=100, train=train, f_permutation=1))
    flow = [dict(f_width=256), dict(f_width=240, nz=4, f_depth=1), dict(f_width=236, nz=4, f_depth=1),
            dict(nz=256, f_permutation=2), dict(nz=232, f_permutation=2, f_width=4, f_depth=1),
            dict(nz=208, f_permutation=2, f_depth=32), dict(nz=256, f_permutation=1, f_width=200, f_depth=1),
            dict(nz=100, f_width=196, f_depth=32), dict(nz=256, f_permutation=1, f_width=64),
            dict(nz=128, f_width=64, f_depth=32, batch=1250), dict(nz=100, f_width=128, f_depth=32, batch=1250),
            dict(nz=4, f_width=232, f_depth=1, batch=33), dict(nz=228, f_permutation=2, f_width=4, f_depth=1),
            dict(nz=204, f_permutation=2, f_depth=32), dict(nz=256, f_permutation=1, f_width=196, f_depth=1),
            dict(nz=100, f_width=192, f_depth=32), dict(nz=200, f_width=100, f_depth=1, f_permutation=1, batch=1203)]
    for kw in flow:                                                     # tests/test_flow_plan_limits.py
        for arch, ngf in ((-1, 0), (0, 64), (1, 128)):
            out.append(config(**dict(dict(arch=arch, ngf=ngf), **kw)))
    bad = dict(arch=[7, -2], batch=[0, -1], nz=[0, 3, 6, 260], ngf=[0, -64, 16, 40], nc=[0, 5],
               f_depth=[0, 33], f_width=[0, 2, 260, 256], f_permutation=[0, 3], f_coupling=[2, -1],
               gemm_impl=[2], bwd_passes=[2, 4])
    singles = [(f, v) for f, vs in bad.items() for v in vs]
    for base in ({}, dict(arch=1, nz=128, ngf=128), dict(arch=3, batch=8, f_width=128), dict(arch=-1, ngf=0)):
        for (f, v), in itertools.combinations(singles, 1):
            out.append(config(**dict(base, **{f: v})))
        for (f1, v1), (f2, v2) in itertools.combinations(singles, 2):
            if f1 != f2:
                out.append(config(**dict(base, **{f1: v1, f2: v2})))
    return out


def record(lib, cfg):
    h = C.c_void_p()
    rc = lib.lsnf_plan_create(C.byref(_cabi.Config(**cfg)), C.byref(h))
    if rc:
        return {"rc": rc, "error": lib.lsnf_last_error().decode()}
    r = {"rc": 0, "ws_bytes": lib.lsnf_workspace_bytes(h), "stages": [], "launch": {},
         "langevin_launches": [lib.lsnf_langevin_launch_count(h, t) for t in (0, 1, 20, 40, 41, 400, 8000)]}
    n = lib.lsnf_plan_num_stages(h)
    for i in range(n):
        s = _cabi.StageInfo()
        _cabi.check(lib.lsnf_plan_stage_info(h, i, C.byref(s)), "stage_info")
        r["stages"].append(flat(s))
    for sms in SMS:
        rows = []
        for i in range(n):
            li = _cabi.LaunchInfo()
            _cabi.check(lib.lsnf_plan_stage_launch_info(h, i, sms, C.byref(li)), "launch_info")
            rows.append(flat(li))
        r["launch"][str(sms)] = rows
    k = cfg["f_depth"] * _cabi.FLOW_PTRS_PER_STEP
    off, size = (C.c_int64 * k)(), (C.c_int64 * k)()
    _cabi.check(lib.lsnf_flow_grad_layout(h, off, size), "flow_grad_layout")
    r["flow_grad"] = [list(off), list(size)]
    if cfg["train"] and n:
        off, size = (C.c_int64 * n)(), (C.c_int64 * n)()
        _cabi.check(lib.lsnf_generator_grad_layout(h, off, size), "generator_grad_layout")
        r["gen_grad"] = [list(off), list(size), lib.lsnf_generator_grad_floats(h)]
    lib.lsnf_plan_destroy(h)
    return r


LAYERS = {"svhn": lambda nz, g: [(nz, 8 * g, 4), (8 * g, 4 * g, 4), (4 * g, 2 * g, 4), (2 * g, 3, 4)],
          "cifar10": lambda nz, g: [(nz, 8 * g, 8), (8 * g, 4 * g, 4), (4 * g, 2 * g, 4), (2 * g, 3, 3)]}


def pack_indices(lib):
    """lsnf_plan_pack_index of every weight element of every stage of a small SVHN and a small CIFAR-10 plan, and of
    the first index past each bound."""
    out = {}
    for arch in LAYERS:
        nz, ngf = 8, 32
        cfg = config(arch=_cabi.ARCH[arch], nz=nz, ngf=ngf, batch=3, train=1)
        h = C.c_void_p()
        _cabi.check(lib.lsnf_plan_create(C.byref(_cabi.Config(**cfg)), C.byref(h)), "create")
        digest = hashlib.sha256()
        r, c = C.c_int64(), C.c_int64()
        fn = lib.lsnf_plan_pack_index
        for i in range(lib.lsnf_plan_num_stages(h)):
            s = _cabi.StageInfo()
            _cabi.check(lib.lsnf_plan_stage_info(h, i, C.byref(s)), "stage_info")
            ci_n, co_n, k = LAYERS[arch](nz, ngf)[s.layer]
            vals = []
            for ci, co, ky, kx in itertools.product(range(ci_n), range(co_n), range(k), range(k)):
                _cabi.check(fn(h, i, ci, co, ky, kx, C.byref(r), C.byref(c)), "pack_index")
                vals.append((r.value, c.value))
            for probe in ((ci_n, 0, 0, 0), (0, co_n, 0, 0), (0, 0, k, 0), (0, 0, 0, k), (-1, 0, 0, 0)):
                vals.append((fn(h, i, *probe, C.byref(r), C.byref(c)), lib.lsnf_last_error()))
            digest.update(repr((i, vals)).encode())
        out[arch] = digest.hexdigest()
        lib.lsnf_plan_destroy(h)
    return out


def main():
    if sys.argv[1] == "dump":
        lib = _cabi.load()
        cfgs = configs()
        recs = [{"config": c, "record": record(lib, c)} for c in cfgs]
        with open(sys.argv[2], "w") as f:
            json.dump({"library": _cabi.LIB_PATH, "plans": recs, "pack_index_sha256": pack_indices(lib)}, f)
        return
    a, b = (json.load(open(p)) for p in sys.argv[2:4])
    diffs = [x["config"] for x, y in zip(a["plans"], b["plans"]) if x != y]
    diffs += ["pack_index"] if a["pack_index_sha256"] != b["pack_index_sha256"] else []
    diffs += ["plan count"] if len(a["plans"]) != len(b["plans"]) else []
    ok = [x["record"] for x in a["plans"] if x["record"]["rc"] == 0]
    summary = {
        "plans": len(a["plans"]), "created": len(ok), "rejected": len(a["plans"]) - len(ok),
        "distinct_errors": sorted({x["record"]["error"] for x in a["plans"] if x["record"]["rc"]}),
        "stage_records": sum(len(r["stages"]) for r in ok),
        "launch_records": sum(len(v) for r in ok for v in r["launch"].values()),
        "pack_index_sha256": a["pack_index_sha256"],
        "dump_sha256": [hashlib.sha256(json.dumps(x["plans"], sort_keys=True).encode()).hexdigest() for x in (a, b)],
        "mismatches": diffs,
    }
    text = json.dumps(summary, indent=1)
    print(text)
    if len(sys.argv) > 4:
        with open(sys.argv[4], "w") as f:
            f.write(text + "\n")
    sys.exit(1 if diffs else 0)


if __name__ == "__main__":
    main()
