"""SURVEY.md §8(f) N1 — the reference's inference driver, UNCHANGED, on this package's classes.

`exp/downscaling.py:_run_impl` (the caller of the hot path) is imported from the reference checkout at test time — it
is never copied — after `compat.install()` has bound `thor.score` / `thor.pipelines` / `model.score` to this package.
What the driver needs besides the hot path is replaced by small stand-ins: `lightning.fabric.Fabric` (launch / print /
to_device / autocast / device / global_rank / world_size / is_global_zero, exp/downscaling.py:27-33,61,96-125,252),
`fire`, and `data.pipeline` (xarray I/O) on synthetic in-memory data.

The driver then runs top to bottom: it unpickles a snapshot written with the REFERENCE's classes
(tests/golden/snapshot_tiny.pkl), moves `snapshot["ema"]` to the device, builds `thor.score.BatchedScoreFunction(...)`
with its keywords, conditions it on its own `select_spatiotemporal` closure with per-variable std tensors, and calls
`pipeline.sample(...)`.  This container has no GPU and the package has no CPU path, so the one device call —
`SDAPipeline.sample` — is intercepted here and its arguments checked (operator recognition included); the same flow
with the real CUDA sampler is `tests/test_gpu_parity.py::test_driver_flow_snapshot_to_guided_sampling`.

Runs where the environment variable C2W_REFERENCE names a checkout of schmidtjonathan/Climate2Weather; skipped
elsewhere.
"""
import contextlib
import importlib.util
import os
import pathlib
import sys
import types

import numpy as np
import pytest
import torch

ROOT = pathlib.Path(__file__).resolve().parents[1]
REF = os.environ.get("C2W_REFERENCE")
REF_DRIVER = pathlib.Path(REF, "exp/downscaling.py") if REF else None

pytestmark = pytest.mark.skipif(REF_DRIVER is None or not REF_DRIVER.exists(),
                                reason="C2W_REFERENCE does not name a reference checkout")


class FakeDS:
    """What the driver does with an xarray.Dataset: to_netcdf, coarsen(...).mean().isel(time=...)."""

    def __init__(self, arr, log):
        self.arr, self.log = arr, log

    def to_netcdf(self, path, encoding=None):
        self.log.append(("to_netcdf", pathlib.Path(path).name, tuple(self.arr.shape), sorted(encoding)))
        np.save(str(path) + ".npy", self.arr)

    def coarsen(self, rlat, rlon):
        L, C, H, W = self.arr.shape
        pooled = self.arr.reshape(L, C, H // rlat, rlat, W // rlon, rlon).mean(axis=(3, 5))
        return FakeDS(pooled, self.log)

    def mean(self):
        return self

    def isel(self, time):
        return FakeDS(self.arr[time], self.log)


def _install_stand_ins(monkeypatch, log, L, C, H, W):
    rng = np.random.default_rng(5)
    truth = rng.standard_normal((L, C, H, W)).astype(np.float32)

    dp = types.ModuleType("data.pipeline")
    dp.load_processed = lambda path, data_vars, start, hours, do_nan_check=True: (
        log.append(("load_processed", path, list(data_vars), start, hours)) or FakeDS(truth[:hours], log))
    dp.normalize_ds = lambda ds, quantile_ds, mode: (log.append(("normalize", mode)) or ds)
    dp.unnormalize_ds = lambda ds, quantile_ds, mode: (log.append(("unnormalize", mode)) or ds)
    dp.ds_to_sorted_np = lambda ds, data_vars: ds.arr
    dp.np_to_ds = lambda arr, reference_ds, data_vars: FakeDS(arr, log)
    data = types.ModuleType("data")
    data.pipeline = dp

    class Fabric:
        def __init__(self, **kw):
            self.kw = kw
            self.device = torch.device("cpu")
            self.global_rank, self.world_size, self.is_global_zero = 0, 1, True

        def launch(self):
            pass

        def print(self, *a, **k):
            pass

        def to_device(self, obj):
            return obj.to(self.device)

        def autocast(self):
            return contextlib.nullcontext()

    lightning = types.ModuleType("lightning")
    lf = types.ModuleType("lightning.fabric")
    lf.Fabric = Fabric
    lightning.fabric = lf
    fire = types.ModuleType("fire")
    fire.Fire = lambda *a, **k: None

    for name, m in (("data", data), ("data.pipeline", dp), ("lightning", lightning), ("lightning.fabric", lf),
                    ("fire", fire)):
        monkeypatch.setitem(sys.modules, name, m)
    for name in ("thor", "thor.score", "thor.pipelines", "model", "model.score", "model.nn", "zuko", "zuko.nn", "util"):
        monkeypatch.delitem(sys.modules, name, raising=False)
    import climate2weather_b200.compat as compat

    compat.install(force=True)
    monkeypatch.setattr(sys.modules["util"], "set_random_seed",
                        lambda seed, rank: torch.manual_seed(seed + rank), raising=False)
    return Fabric, truth


def test_unchanged_reference_driver_runs_on_this_package(tmp_path, monkeypatch):
    import climate2weather_b200 as c2w
    from climate2weather_b200 import score as c2w_score

    L, C, H, W = 9, 4, 16, 16  # snapshot_tiny: 12 = 3 frames x 4 variables -> window 3, markov order 1
    log = []
    Fabric, truth = _install_stand_ins(monkeypatch, log, L, C, H, W)

    calls = []

    def fake_sample(self, score_fn, noise, steps=64, corrections=0, tau=1.0, show_progressbar=True, **kw):
        calls.append(dict(pipeline=self, score_fn=score_fn, noise=noise, steps=steps, corrections=corrections, tau=tau,
                          show_progressbar=show_progressbar, extra=kw))
        return torch.full_like(noise, 0.25)

    monkeypatch.setattr(c2w.SDAPipeline, "sample", fake_sample)

    spec = importlib.util.spec_from_file_location("_ref_downscaling", REF_DRIVER)
    drv = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(drv)  # the reference file itself, not a copy

    out = drv._run_impl(
        Fabric(), save_path=tmp_path, model_path=str(ROOT / "tests" / "golden" / "snapshot_tiny.pkl"),
        data_path="cosmo.zarr", quantile_path="q.nc", start_time="2010-01-01", num_hours=L, data_norm_mode="quant99",
        use_exact_grad=False, observation_path="cosmo.zarr", num_sampling_steps=7, num_samples=2, num_corrections=1,
        likelihood_std=[0.1, 0.2, 0.3, 0.4], likelihood_gamma=1e-3, correction_tau=0.3, seed=3, t_step=3, s_step=8,
        batch_size=5)
    assert out == tmp_path

    # two samples, each through SDAPipeline.sample with the driver's keywords
    assert len(calls) == 2
    for c in calls:
        assert isinstance(c["pipeline"], c2w.SDAPipeline) and c["pipeline"].eta == 1e-3
        assert (c["steps"], c["corrections"], c["tau"], c["show_progressbar"], c["extra"]) == (7, 1, 0.3, True, {})
        assert c["noise"].shape == (L, C, H, W) and c["noise"].device.type == "cpu"
        sf = c["score_fn"]
        assert isinstance(sf, c2w.BatchedScoreFunction) and sf.is_conditioned
        assert sf.markov_order == 1 and sf.batch_size == 5
        assert isinstance(sf.unet, c2w.ScoreUNet) and not sf.unet.training
        lk = sf.likelihood
        assert lk["exact"] is False and lk["gamma"] == 1e-3
        # the driver's own closure (AvgPool2d(s)(x[..., ::t, :, :, :])) is recognised as the fused operator family
        op = c2w_score._recognise_operator(lk["A"], L, C, H, W, lk["y"].shape)
        assert (op.t_step, op.s_step) == (3, 8)
        assert c2w_score._per_channel(lk["std"], C, "std") == pytest.approx([0.1, 0.2, 0.3, 0.4])
        want_y = torch.nn.functional.avg_pool2d(torch.from_numpy(truth)[::3], 8, stride=8)
        assert torch.allclose(lk["y"], want_y)

    # what the driver wrote: ground truth, the observation it derived, one file per sample holding sample() output
    written = [e for e in log if e[0] == "to_netcdf"]
    assert [e[1] for e in written] == ["ground_truth.nc", "observation.nc", "gen_sample_000.nc", "gen_sample_001.nc"]
    assert written[1][2] == (3, C, 2, 2) and written[2][2] == (L, C, H, W)
    got = np.load(str(tmp_path / "gen_sample_001.nc") + ".npy")
    assert got.dtype == np.float32 and np.all(got == 0.25)
