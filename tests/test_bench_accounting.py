"""bench.py's ALGORITHMIC work per latent-step -- the numerator of `roofline.achieved` and of
`frac_of_tensor_roofline` -- is the figure SURVEY.md section 8(d) states: 2 x the generator's exact forward FLOPs (taps
that land inside the output; forward + data gradient, ONE pass each) + the flow term; extra split-precision passes and
zero-filled border taps never count.  Also: the library's nominal per-stage FLOPs are torch FlopCounter's."""
import ctypes as C

import pytest

import bench
from lsnf_b200 import _cabi, synth

# SURVEY.md section 8(a) layer table, "exact MFLOP" column, and section 8(d) "ALGORITHMIC work per latent-step"
EXACT_MFLOP = {
    "svhn": [1.64, 51.38, 58.98, 2.95],
    "cifar10": [16.78, 943.72, 1007.68, 13.57],
    "celeba_crop": [3.28, 205.52, 235.93, 251.92, 12.19],
    "celeba_hq256": [6.55, 822.08, 943.72, 1007.68, 1040.45, 2114.06, 199.76],
}
NOMINAL_MFLOP = {"svhn": 139.0, "cifar10": 2178.4, "celeba_crop": 821.2, "celeba_hq256": 6650.3}
ALG_GFLOP_PER_LATENT_STEP = {"svhn": 0.2304, "cifar10": 3.9641, "celeba_crop": 1.4181, "celeba_hq256": 12.2695}
FLOW_MFLOP = {"svhn": 0.474, "cifar10": 0.655, "celeba_crop": 0.474, "celeba_hq256": 0.912}


@pytest.mark.parametrize("name", sorted(bench.WORKLOADS))
def test_algorithmic_flops_are_the_survey_figures(name):
    w = bench.WORKLOADS[name]
    layers = synth.generator_layers(w["dataset"], w["nz"], w["ngf"])
    exact = bench.exact_layer_flops(layers)
    assert [round(e / 1e6, 2) for e in exact] == EXACT_MFLOP[name]
    flow = bench.flow_flops(w["nz"], w["f_width"])
    assert flow / 1e6 == pytest.approx(FLOW_MFLOP[name], abs=6e-4)
    alg = 2.0 * sum(exact) + flow
    assert alg / 1e9 == pytest.approx(ALG_GFLOP_PER_LATENT_STEP[name], abs=1e-4)
    # the roofline table of BASELINE.md section 3 (latent-steps/s at 100 % of the sustained bf16 peak) follows from it
    assert 1376.8e12 / alg == pytest.approx(bench.ROOFLINE_LATENT_STEPS[name], rel=5e-3)


@pytest.mark.parametrize("name", sorted(bench.WORKLOADS))
def test_library_stage_flops_are_nominal_and_never_below_the_algorithmic_ones(name):
    w = bench.WORKLOADS[name]
    lib = _cabi.load()
    cfg = _cabi.Config(arch=_cabi.ARCH[w["dataset"]], batch=w["B"], nz=w["nz"], ngf=w["ngf"], nc=3, f_depth=5,
                       f_width=w["f_width"], f_permutation=2, f_coupling=1, leak=0.2, gemm_impl=0, bwd_passes=3, train=0)
    h = C.c_void_p()
    _cabi.check(lib.lsnf_plan_create(C.byref(cfg), C.byref(h)), "lsnf_plan_create")
    try:
        layers = synth.generator_layers(w["dataset"], w["nz"], w["ngf"])
        exact = bench.exact_layer_flops(layers)
        n = lib.lsnf_plan_num_stages(h)
        assert n == 2 * len(layers)
        fwd_nominal = 0.0
        for i in range(n):
            info = _cabi.StageInfo()
            _cabi.check(lib.lsnf_plan_stage_info(h, i, C.byref(info)), "lsnf_plan_stage_info")
            assert info.passes == 3
            # what the tensor pipe is asked to do (padding of K / N tiles and zero-filled taps included) is never
            # less than the algorithmic work the roofline claim counts
            assert info.flops >= exact[info.layer] * w["B"] * (1 - 1e-9)
            if info.kind == 0:
                fwd_nominal += info.flops / w["B"]
        # hidden layers are counted exactly as torch.utils.flop_counter does (2 H_in^2 C_in C_out k^2); the first and
        # last layers carry K / N padding on top, so the sum is bounded below by the FlopCounter figure
        assert fwd_nominal / 1e6 >= NOMINAL_MFLOP[name] * (1 - 1e-3)
        assert fwd_nominal / 1e6 <= NOMINAL_MFLOP[name] * 1.35
    finally:
        lib.lsnf_plan_destroy(h)


def test_reference_arm_times_one_whole_training_iteration_of_config_1():
    """`bench.py --impl reference --mode train --workload svhn`: BASELINE.json's config 1 ("one training iteration on
    CPU: flow prior + short-run Langevin + generator update") on the host cores, same JSON contract as the CUDA arm's
    `--mode train` line."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--mode", "train",
                        "--workload", "svhn", "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "train_iteration_latent_steps_per_sec"
    assert line["mode"] == "train" and line["gpu_launches"] == 0 and line["higher_is_better"] is True
    assert line["config"] == bench.workload_config("svhn", bench.WORKLOADS["svhn"])
    d = line["details"]
    assert d["ms_per_iteration"] == pytest.approx(d["langevin_call_ms"] + d["updates_ms"], rel=1e-9)
    assert line["value"] == pytest.approx(100 * 20 / (d["ms_per_iteration"] * 1e-3), rel=1e-9)
    assert d["langevin_call_ms"] > d["updates_ms"] > 0           # SURVEY section 6: 1 467 ms against 110 ms on 8 vCPU
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": "latent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones_the_same_way(tmp_path):
    import numpy as np
    import torch
    n = bench.DUMP_MAX_ELEMENTS
    arrays = {"small": torch.arange(6, dtype=torch.float16).reshape(2, 3), "f64": torch.ones(3, dtype=torch.float64),
              "big": torch.arange(n + 1000, dtype=torch.int32)}
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    small, f64, big = (np.load(tmp_path / "a" / f"{k}.npy") for k in ("small", "f64", "big"))
    assert small.dtype == np.float32 and small.shape == (2, 3) and np.array_equal(small, np.arange(6).reshape(2, 3))
    assert f64.dtype == np.float64
    assert big.dtype == np.float32 and big.shape == (n,) and np.all(np.diff(big) > 0) and big[-1] < n + 1000
    assert np.array_equal(big, np.load(tmp_path / "b" / "big.npy"))


@pytest.mark.gpu
def test_steps_are_timed_calls_and_the_dump_is_the_last_one(tmp_path):
    """`--steps K --warmup W` times K Langevin calls, call i with Philox seed 1234 + W + i, and --dump-outputs writes
    what the last of them returned: what the public API returns for that seed."""
    import json
    import subprocess
    import sys
    import numpy as np
    import torch
    import lsnf_b200
    from helpers import rel_l2
    r = subprocess.run([sys.executable, bench.__file__, "--workload", "svhn", "--steps", "2", "--warmup", "3",
                        "--no-cpu-baseline", "--no-secondary", "--no-eager-ref", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["details"]["langevin_calls_per_step"] == 1
    w = bench.WORKLOADS["svhn"]
    dev = torch.device("cuda:0")
    args, netG, netF, _, _ = bench.build_models(w, dev)
    x_np, z0_np, _ = synth.inputs(w["B"], w["nz"], 3, w["img"], 1, seed=1)
    z, gn, fn = lsnf_b200.sample_langevin_post_z_with_flow(torch.from_numpy(z0_np).to(dev), torch.from_numpy(x_np).to(dev),
                                                           netG, netF, args, seed=1234 + 3 + 1, steps=w["T"])
    z_T = np.load(tmp_path / "z_T.npy")
    assert z_T.dtype == np.float32 and z_T.shape == (w["B"], w["nz"])
    assert rel_l2(z_T, z.reshape(w["B"], w["nz"]).cpu().numpy()) < 1e-6
    assert float(np.load(tmp_path / "gnorm_g.npy")) == pytest.approx(gn.item(), rel=1e-6)
    assert float(np.load(tmp_path / "gnorm_f.npy")) == pytest.approx(fn.item(), rel=1e-6)


@pytest.mark.gpu
def test_train_mode_dump_is_the_last_timed_iteration(tmp_path):
    """`--mode train --steps 1 --warmup 3`: three warm-up iterations (seeds 1000-1002), one timed one (seed 1100),
    then more iterations for the other rows.  The dump holds the timed iteration's results and the parameters it left:
    the same as replaying those four iterations here, and the losses the JSON line reports."""
    import json
    import os
    import subprocess
    import sys
    import numpy as np
    import torch
    import lsnf_b200
    from helpers import rel_l2
    r = subprocess.run([sys.executable, bench.__file__, "--mode", "train", "--workload", "svhn", "--steps", "1",
                        "--warmup", "3", "--dump-outputs", str(tmp_path / "bench")],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])["details"]
    assert d["training_iterations_per_step"] == 1
    assert float(np.load(tmp_path / "bench" / "loss_g.npy")) == d["loss_g"]
    assert float(np.load(tmp_path / "bench" / "loss_f.npy")) == d["loss_f"]
    w = bench.WORKLOADS["svhn"]
    dev = torch.device("cuda:0")
    args, netG, netF, _, _ = bench.build_models(w, dev)
    optG, optF = lsnf_b200.make_optimizers(netG, netF, args)
    x = torch.from_numpy(synth.inputs(w["B"], w["nz"], 3, w["img"], 1, seed=1)[0]).to(dev)
    for seed in (1000, 1001, 1002, 1100):
        lg, lf, gn, fn, zk = lsnf_b200.training_iteration(x, netG, netF, optG, optF, args, global_batch=w["B"],
                                                          sample_offset=0, seed=seed)
    bench.dump_outputs(str(tmp_path / "here"), {
        "loss_g": lg, "loss_f": lf, "gnorm_g": gn, "gnorm_f": fn, "z_k": zk,
        "generator_params": torch.cat([p.detach().reshape(-1) for p in netG.parameters()]),
        "flow_params": torch.cat([p.detach().reshape(-1) for p in netF.parameters()])})
    names = sorted(os.listdir(tmp_path / "bench"))
    assert names == sorted(os.listdir(tmp_path / "here")) and len(names) == 7
    for f in names:
        got, want = np.load(tmp_path / "bench" / f), np.load(tmp_path / "here" / f)
        assert got.dtype == np.float32 and got.shape == want.shape, f
        assert rel_l2(got, want) < 1e-5, (f, rel_l2(got, want))


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    import subprocess
    import sys
    r = subprocess.run([sys.executable, bench.__file__, "--impl", "reference", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
