"""The kernels each host entry queues, counted exactly: RsBatchStats.kernel_launches and groups of
roadsurf_run_batch and roadsurf_run_host_soa, and the RsLaunchInfo they leave behind.  Every expected
number is the sum of the launches the entry makes:

- roadsurf_run_batch, per group of points with one time axis: the solar table, then per device batch one
  forcing transpose and one output transpose per staging chunk (one chunk at these sizes), and the model run;
- roadsurf_run_host_soa: the solar table, then per column chunk of 65 536 points the sky-view partition when
  the entry builds the point order itself (coarse records with horizons and no prepared statics), and the
  model run;
- a model run is one step-kernel launch, or 2 * passes + 3 with coupling lane compaction: the window, per
  pass a partition and a compacted pass, then a final partition and the rest of the run.
"""
import numpy as np
import pytest

from roadsurf_b200 import synth

pytestmark = pytest.mark.gpu


def _batch(rslib, arrays, settings, params):
    before = rslib.last_launch()["launches_total"]
    rslib.run_batch(arrays, settings, params)
    st, li = rslib.last_batch_stats(), rslib.last_launch()
    assert li["launches_total"] - before == st["kernel_launches"]
    assert li["nlayers"] == settings.NLayers and li["forcing_mode"] == 0
    return st["kernel_launches"], st["groups"]


def test_run_batch_launches(rslib):
    arrays, settings, params, _ = synth.make_case(100, 6, seed=501)
    assert _batch(rslib, arrays.copy(), settings, params) == (4, 1)         # solar, transpose in, model, transpose out
    rslib.set_option("max_points_per_device_batch", 64)                     # 128 slots -> two device batches
    try:
        assert _batch(rslib, arrays.copy(), settings, params) == (1 + 2 * 3, 1)
    finally:
        rslib.set_option("max_points_per_device_batch", 0)


def test_run_batch_launches_with_coupling_compaction(rslib):
    arrays, settings, params, _ = synth.make_case(300, 4, seed=48, analysis_hours=4, use_coupling=1, use_relaxation=1,
                                                  settings_kw=dict(coupling_minutes=120))
    try:
        for passes in (6, 2):
            rslib.set_option("coupling_compaction_passes", passes)
            assert _batch(rslib, arrays.copy(), settings, params) == (3 + 2 * passes + 3, 1), passes
        rslib.set_option("coupling_compaction_passes", 0)                   # one launch, warps repeat the window
        assert _batch(rslib, arrays.copy(), settings, params) == (4, 1)
    finally:
        rslib.set_option("coupling_compaction_passes", 6)


def _host_soa(rslib, settings, params, h, forcing_mode, **kw):
    n_out = (h["tf"].shape[1] + 119) // 120
    npts = h["local"].shape[1]
    out = np.zeros((rslib.O_NVAR, n_out, npts))
    rslib.run_host_soa(settings, params, h["forcing"], h["tf"], h["local"], out, out_stride=120,
                       record_step=h["rs"] if forcing_mode == 1 else None, **kw)
    st, li = rslib.last_batch_stats(), rslib.last_launch()
    assert li["nlayers"] == settings.NLayers and li["forcing_mode"] == forcing_mode
    return st["kernel_launches"], st["groups"]


def _soa_arrays(db, idx):
    return dict(forcing=db.forcing[:, :, idx].cpu().numpy(), local=db.local[:, idx].cpu().numpy(),
                hor=db.horizons[:, idx].cpu().numpy(), tf=db.time_fields.cpu().numpy(),
                rs=None if db.record_step is None else db.record_step.cpu().numpy())


def test_host_soa_launches_full_resolution(rslib):
    import torch
    arrays, settings, params, _ = synth.make_case(1000, 6, seed=502)
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(1000, arrays.sim_len, horizons=True)
    db.load_point_arrays(arrays)
    h = _soa_arrays(db, torch.arange(1000, device="cuda"))
    assert _host_soa(rslib, settings, params, h, 0, horizons=h["hor"]) == (2, 1)     # solar, model
    handle = rslib.prepare_statics(h["local"], h["hor"])
    try:
        assert _host_soa(rslib, settings, params, h, 0, statics=handle) == (2, 1)
    finally:
        rslib.release_statics(handle)


def test_host_soa_launches_coarse_records(rslib):
    import torch
    npts = 70000 + 5                                                        # two column chunks
    arrays, settings, params, rec = synth.make_case(256, 6, seed=503)
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(256, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True)
    db.load_records(rec)
    db.time_fields.copy_(torch.from_numpy(arrays.time))
    db.load_local(arrays.local, arrays.local_horizons)
    h = _soa_arrays(db, (torch.arange(npts, device="cuda") * 7) % 256)
    assert _host_soa(rslib, settings, params, h, 1) == (1 + 2, 2)                       # no horizons: no partition
    assert _host_soa(rslib, settings, params, h, 1, horizons=h["hor"]) == (1 + 2 * 2, 2)  # partition + model per chunk
    handle = rslib.prepare_statics(h["local"], h["hor"])
    try:
        assert _host_soa(rslib, settings, params, h, 1, statics=handle) == (1 + 2, 2)   # the prepared order
    finally:
        rslib.release_statics(handle)


def test_host_soa_launches_with_coupling_compaction(rslib):
    import torch
    arrays, settings, params, rec = synth.make_case(777, 5, seed=49, analysis_hours=3, use_coupling=1,
                                                    use_relaxation=1, obs_bias=False,
                                                    settings_kw=dict(coupling_minutes=60))
    rslib.set_model(settings, params)
    db = rslib.DeviceBatch(777, arrays.sim_len, n_records=rec.nrec, coarse=True, horizons=True, coupling=True)
    db.load_records(rec)
    db.time_fields.copy_(torch.from_numpy(arrays.time))
    db.load_local(arrays.local, arrays.local_horizons)
    h = _soa_arrays(db, torch.arange(777, device="cuda"))
    wend = arrays.local[0].couplingIndexI
    assert _host_soa(rslib, settings, params, h, 1, horizons=h["hor"]) == (3, 1)
    assert _host_soa(rslib, settings, params, h, 1, horizons=h["hor"], coupling_window_end=wend) == (2 + 2 * 6 + 3, 1)
