"""Host-side pieces of bench.py that need no GPU: the one-poller-per-job clock sampler (against a stand-in NVML), the config dict
both arms print, the timed loop (against a stand-in column), --dump-outputs, and the steps of the configs' CPU arm."""
import importlib
import json
import sys
import time
import types

import numpy as np
import pytest


@pytest.fixture()
def bench(monkeypatch):
    fake = types.ModuleType("pynvml")
    fake.NVML_CLOCK_SM = 1
    fake.nvmlClocksEventReasonSwPowerCap = 0x4
    fake.nvmlClocksEventReasonHwSlowdown = 0x8
    fake.nvmlClocksEventReasonSwThermalSlowdown = 0x20
    fake.nvmlClocksEventReasonHwThermalSlowdown = 0x40
    fake.nvmlClocksEventReasonHwPowerBrakeSlowdown = 0x80
    fake.calls = []
    fake.nvmlInit = lambda: None
    fake.nvmlDeviceGetHandleByIndex = lambda i: ("gpu", i)
    fake.nvmlDeviceGetMaxClockInfo = lambda h, k: 1965
    fake.nvmlDeviceGetClockInfo = lambda h, k: 1965 - 15 * h[1]
    fake.nvmlDeviceGetCurrentClocksEventReasons = lambda h: 0x4 if h[1] == 2 else 0
    monkeypatch.setitem(sys.modules, "pynvml", fake)
    sys.modules.pop("bench", None)
    return importlib.import_module("bench")


def test_rank0_watches_every_gpu_and_other_ranks_do_not_poll(bench, monkeypatch):
    monkeypatch.delenv("CUDA_VISIBLE_DEVICES", raising=False)
    s = bench.ClockSampler([0, 1, 2, 3])
    assert s.ok and len(s.handles) == 4
    t0 = time.perf_counter()
    s.start()
    time.sleep(0.05)
    s.stop_flag = True
    s.join(timeout=1)
    out = s.summary(t0, time.perf_counter())
    assert out["samples"] >= 3 and out["gpus_watched"] == 4
    assert out["sm_mhz_per_gpu"] == [1965.0, 1950.0, 1935.0, 1920.0] and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"]          # GPU 2's reason is reported for the job
    idle = bench.ClockSampler([])
    idle.start(); idle.join(timeout=1)
    assert not idle.ok and idle.summary(0, 1)["sm_mhz"] is None


def test_nvml_index_follows_cuda_visible_devices(bench, monkeypatch):
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "4,5,7")
    assert [bench._nvml_index(i) for i in range(4)] == [4, 5, 7, 3]
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "GPU-8f6d")
    assert bench._nvml_index(1) == 1
    s = bench.ClockSampler([0])
    assert s.ok


def test_both_arms_print_the_same_config(bench):
    """The driver compares the `config` of the two arms: one function makes it, keyed only by the GPU count and the series."""
    for n in (1, 2, 8):
        for series in ("weak", "strong"):
            c = bench.config_dict(n, series)
            assert c == bench.config_dict(n, series) and c["n_gpus"] == n and c["scaling"] == series
            assert "workload" in c and "model" not in c
    assert bench.config_dict(1, "weak")["rows"] == 100_000_000


def test_timed_loop_runs_steps_and_keeps_the_last_output(bench):
    """timed_loop runs exactly --steps steps; with keep_last the last one's c stays allocated for --dump-outputs, every other c
    is freed, and loop.last is that step's result."""
    made = []

    class Col:
        freed = False

        def free(self):
            self.freed = True

    class Fut:
        def __init__(self, i):
            self.i = i

        def result(self):
            return {"sum": float(self.i), "count": self.i, "rows": self.i}

    class Src:
        def binary_agg_async(self, op, other):
            made.append(Col())
            return made[-1], Fut(len(made) - 1)

    ctx = types.SimpleNamespace(comm_barrier=lambda: None, timer_start=lambda: None, timer_stop=lambda: 1.0)
    loop = bench.HotLoop(types.SimpleNamespace(ADD=0), Src(), None, depth=1)
    assert bench.timed_loop(ctx, loop, 7, 1, keep_last=True) == 1.0
    assert len(made) == 7 and loop.last == (6.0, 6, 6)
    assert loop.last_c is made[-1] and not made[-1].freed and all(c.freed for c in made[:-1])
    bench.timed_loop(ctx, loop, 3, 1)
    assert len(made) == 10 and all(c.freed for c in made[7:])


def test_dump_outputs_writes_the_same_rows_every_run(bench, tmp_path):
    rng = np.random.default_rng(3)
    small = [rng.uniform(-1, 1, n) for n in (1000, 5, 300)]
    big = [rng.uniform(-1, 1, bench.DUMP_ROWS) for _ in range(2)]
    for d, chunks in (("a", small), ("b", small), ("big", big)):
        bench.dump_outputs(str(tmp_path / d), chunks, 1.5, 7)
    for f in ("c.npy", "sum.npy", "count.npy"):
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype == np.float64 and np.array_equal(x, y), f
    c = np.load(tmp_path / "a" / "c.npy")
    assert c.shape == (1305,) and np.isin(c, np.concatenate(small)).all()
    assert np.load(tmp_path / "a" / "sum.npy").tolist() == [1.5] and np.load(tmp_path / "a" / "count.npy").tolist() == [7.0]
    assert np.load(tmp_path / "big" / "c.npy").shape == (bench.DUMP_ROWS,)
    assert sum(p.stat().st_size for p in (tmp_path / "big").iterdir()) <= 64 << 20


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--config", "3", "--dump-outputs", "out"], ["--config", "5", "--steps", "0"],
                                  ["--config", "4", "--impl", "reference", "--steps", "-1"]])
def test_bench_rejects_arguments_it_cannot_honour(bench, monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit):
        bench.main()


def test_config_reference_arm_times_steps_passes(bench, oracle, monkeypatch, capsys):
    """The configs' CPU arm runs --warmup untimed and --steps timed passes of the oracle and reports --steps."""
    from benchmarks import configs_bench

    passes = []
    real = oracle.aggregate
    monkeypatch.setattr(oracle, "aggregate", lambda *a: passes.append(1) or real(*a))   # config 4: one sum per pass
    args = types.SimpleNamespace(config=4, steps=3, warmup=2, gpus=1, scaling="strong")
    configs_bench.reference_arm(args, 0)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert len(passes) == 5 and line["steps"] == 3 and line["warmup"] == 2 and line["value"] > 0
