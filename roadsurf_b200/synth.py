"""Seeded synthetic road-weather inputs for the BASELINE.json configurations (SURVEY.md section 8d).

Hourly records are drawn per point and then interpolated to the model time step exactly as the
reference's example does (examples/example1/src/JsonSource.cpp:49-176): linear in time,
`a + (t - t_a) * (b - a) / (t_b - t_a)` with integer seconds, precipitation phase taken from the
NEXT record.  The same record arrays feed the coarse-forcing device path, which performs that
interpolation on the GPU.
"""
import datetime as _dt
import math

import numpy as np

from . import abi

SIGMA = 5.67e-8
FORECAST_START = _dt.datetime(2019, 12, 2, 0, 0, 0)  # RoadSurfUserManual.pdf section 5.1

RECORD_VARS = ("tair", "tdew", "VZ", "Rhz", "prec", "SW", "LW", "SW_dir", "LW_net", "TSurfObs",
               "PrecPhase")


def time_axis(start, sim_len, dt_secs):
    """int32 [6, sim_len]: year, month, day, hour, minute, second of every model step."""
    out = np.empty((6, sim_len), dtype=np.int32)
    step = _dt.timedelta(seconds=dt_secs)
    t = start
    for i in range(sim_len):
        out[:, i] = (t.year, t.month, t.day, t.hour, t.minute, t.second)
        t = t + step
    return out


def tdew_from_rh(t, rh):
    """examples/example1/src/MeteorologyTools.cpp:12-51 (RH -> dew point branch)."""
    alpha = np.where(t >= 0.0, 17.269, 21.875)
    beta = np.where(t >= 0.0, 237.3, 265.5)
    afact = 0.61078
    esat = afact * np.exp(alpha * t / (t + beta))
    epr = 0.01 * rh * esat
    xx = np.log(epr / afact)
    return beta * xx / (alpha - xx)


def _solar_elevation_deg(when, lat_deg, lon_deg):
    """Plain declination / hour-angle elevation (synthetic SW only; not the model's Meeus code)."""
    doy = when.timetuple().tm_yday
    decl = math.radians(-23.44) * math.cos(2.0 * math.pi * (doy + 10) / 365.0)
    hours = when.hour + when.minute / 60.0 + when.second / 3600.0
    ha = np.radians(15.0 * (hours - 12.0) + lon_deg)
    lat = np.radians(lat_deg)
    s = np.sin(lat) * math.sin(decl) + np.cos(lat) * math.cos(decl) * np.cos(ha)
    return np.degrees(np.arcsin(np.clip(s, -1.0, 1.0)))


class Records:
    """Hourly (coarse) forcing records for a batch of points: arrays [npoints, nrec]."""

    def __init__(self, npoints, nrec):
        self.npoints, self.nrec = npoints, nrec
        for v in RECORD_VARS:
            setattr(self, v, np.zeros((npoints, nrec)))
        self.lat = np.zeros(npoints)
        self.lon = np.zeros(npoints)
        self.sky_view = np.ones(npoints)
        self.horizons = np.zeros((npoints, 360))
        self.record_step = np.zeros(nrec, dtype=np.int32)  # 0-based model step of every record
        self.obs_bias = None  # optional [npoints, 3]: analysis-period offsets of tair, VZ, Rhz


def draw_records(npoints, nrec, seed, start, record_secs=3600, dt_secs=30.0, first_step=0,
                 sky_view_fraction=0.3, phase_missing_fraction=0.5, member_perturbation=None):
    """Draw `nrec` records spaced `record_secs` apart, the first at model step `first_step`."""
    rng = np.random.Generator(np.random.PCG64(seed))
    r = Records(npoints, nrec)
    per = int(round(record_secs / dt_secs))
    r.record_step[:] = first_step + per * np.arange(nrec, dtype=np.int32)
    r.lat[:] = rng.uniform(59.8, 69.9, npoints)
    r.lon[:] = rng.uniform(20.0, 31.0, npoints)
    obstructed = rng.random(npoints) < sky_view_fraction
    r.sky_view[:] = np.where(obstructed, rng.uniform(0.4, 1.0, npoints), 1.0)
    # smooth horizon profile: 8 deg * |low-pass noise| for obstructed points
    k = rng.standard_normal((npoints, 6))
    ang = np.radians(np.arange(360.0))
    prof = sum(k[:, [j]] * np.cos((j + 1) * ang[None, :] + j) for j in range(6)) / math.sqrt(6.0)
    r.horizons[:] = np.where(obstructed[:, None], 8.0 * np.abs(prof), 0.0)

    t0 = rng.normal(-1.0, 3.0, npoints)
    amp = rng.uniform(1.0, 5.0, npoints)
    noise = np.zeros((npoints, nrec))
    x = rng.normal(0.0, 1.0, npoints)
    for j in range(nrec):
        x = 0.8 * x + rng.normal(0.0, 0.6, npoints)
        noise[:, j] = x
    cloud = rng.uniform(0.2, 1.0, (npoints, nrec))
    rh_noise = rng.standard_normal((npoints, nrec))
    vz = np.clip(rng.lognormal(math.log(3.0), 0.6, (npoints, nrec)), 0.0, 25.0)
    wet = rng.random((npoints, nrec)) < 0.15
    amount = rng.exponential(0.8, (npoints, nrec))
    lw_noise = rng.normal(0.0, 15.0, (npoints, nrec))
    phase_missing = rng.random(npoints) < phase_missing_fraction
    obs_noise = rng.normal(0.0, 0.5, (npoints, nrec))

    if member_perturbation is not None:
        mrng = np.random.Generator(np.random.PCG64(seed * 1000003 + member_perturbation))
        t0 = t0 + mrng.normal(0.0, 1.0, npoints)
        amount = amount * mrng.lognormal(0.0, 0.3, (npoints, nrec))
        cloud = np.clip(cloud * mrng.uniform(0.8, 1.2, (npoints, nrec)), 0.05, 1.0)

    for j in range(nrec):
        when = start + _dt.timedelta(seconds=float(r.record_step[j]) * dt_secs)
        hour = when.hour + when.minute / 60.0
        tair = t0 + amp * math.sin(2.0 * math.pi * (hour - 15.0) / 24.0) + noise[:, j]
        r.tair[:, j] = tair
        r.Rhz[:, j] = np.clip(88.0 + 8.0 * rh_noise[:, j], 35.0, 100.0)
        elev = _solar_elevation_deg(when, r.lat, r.lon)
        sw = np.maximum(0.0, 1361.0 * 0.7 * np.sin(np.radians(elev))) * cloud[:, j]
        r.SW[:, j] = sw
        r.SW_dir[:, j] = 0.6 * sw
        lw = np.clip(0.80 * SIGMA * (tair + 273.15) ** 4 + lw_noise[:, j], 100.0, 450.0)
        r.LW[:, j] = lw
        r.LW_net[:, j] = lw - 0.95 * SIGMA * (tair + 272.15) ** 4
        given = np.where(tair < -0.5, 3.0, np.where(tair < 1.0, 2.0, 1.0))
        r.PrecPhase[:, j] = np.where(phase_missing, -9999.0, given)
        r.TSurfObs[:, j] = tair - 1.0 + obs_noise[:, j]
    r.tdew[:] = tdew_from_rh(r.tair, r.Rhz)
    r.VZ[:] = vz
    r.prec[:] = np.where(wet, amount, 0.0)
    return r


def interpolate_records(rec, sim_len, dt_secs=30.0):
    """Records -> per-step arrays, following JsonSource.cpp:49-176 for a record grid that starts
    at or before step 0.  Steps at or after the LAST record are left missing, as the reference's loop
    leaves them (`rawPos+1<rawLen`, JsonSource.cpp:85).  Times are integer seconds there, so the
    weights are formed from seconds, not steps (the rounding differs).  Returns dict name ->
    [npoints, sim_len] (PrecPhase as int32)."""
    steps = np.arange(sim_len, dtype=np.int64)
    rs = rec.record_step.astype(np.int64)
    if rs[0] > 0:
        raise ValueError("the first record must lie at or before step 0")
    beyond = steps >= rs[-1]
    k = np.minimum(np.searchsorted(rs, steps, side="right") - 1, len(rs) - 2)  # rs[k] <= step < rs[k+1]
    dt_a = (steps - rs[k]).astype(np.float64) * dt_secs
    span = (rs[k + 1] - rs[k]).astype(np.float64) * dt_secs
    exact = (steps == rs[k])
    out = {}
    for v in RECORD_VARS:
        a = getattr(rec, v)[:, k]
        b = getattr(rec, v)[:, k + 1]
        if v == "PrecPhase":
            val = np.where(exact[None, :], a, b)
            out[v] = np.where((val > -100.0) & ~beyond[None, :], val, -9999.0).astype(np.int32)
            continue
        miss = -1000.0 if v == "LW_net" else -100.0
        interp = a + (dt_a[None, :] * (b - a)) / span[None, :]
        ok_between = (a > miss) & (b > miss)
        val = np.where(exact[None, :], np.where(a > miss, a, -9999.9),
                       np.where(ok_between, interp, -9999.9))
        out[v] = np.where(beyond[None, :], -9999.9, val)
    return out


def read_input_derive(arrays, settings, forecast_step):
    """What examples/example1/src/roadrunner.cpp:157-278 (read_input) derives per point.

    `forecast_step` is the number of model steps between simulation start and forecast start
    (init_secs / DTSecs).  Fills arrays.local[p] and blanks TSurfObs over the coupling window.
    """
    npoints, sim_len = arrays.npoints, arrays.sim_len
    span = int(settings.coupling_minutes * 60 / settings.DTSecs)
    for p in range(npoints):
        lp = arrays.local[p]
        lp.InitLenI = 1 + int(forecast_step)
        if settings.use_relaxation == 1:
            lp.tair_relax = lp.VZ_relax = lp.RH_relax = -9999.9
            # GetLatestObsIndex (JsonSource.cpp:397-414): 1-based count of observed steps, or
            # -9999 when the point has no observations at all
            last = int(forecast_step) + 1 if forecast_step > 0 else -9999
            if last > -1 and last < sim_len:
                lp.InitLenI = last
                lp.tair_relax = arrays.tair[p, last]
                lp.VZ_relax = arrays.VZ[p, last]
                lp.RH_relax = arrays.Rhz[p, last]
        if settings.use_coupling == 1:
            lp.couplingTsurf = -9999.9
            lp.couplingIndexI = -9999
            obs = arrays.TSurfObs[p]
            i = sim_len - 1
            while i >= 0 and (np.isnan(obs[i]) or obs[i] < -100.0):
                i -= 1
            if i >= span:
                lp.couplingTsurf = obs[i]
                lp.couplingIndexI = i
                obs[i - span + 1:i + 1] = -9999.9


def case_from_records(rec, hours, analysis_hours=0, use_coupling=0, use_relaxation=0, dt=30.0, nlayers=15,
                      start=None, **settings_kw):
    """Full-resolution host-layout case built deterministically (no random numbers) from coarse
    records: (PointArrays, InputSettings, InputParameters)."""
    start = start or FORECAST_START
    npoints = rec.npoints
    per_hour = int(round(3600.0 / dt))
    sim_len = 1 + (analysis_hours + hours) * per_hour
    sim_start = start - _dt.timedelta(hours=analysis_hours)
    forecast_step = analysis_hours * per_hour
    fields = interpolate_records(rec, sim_len, dt)
    pa = abi.PointArrays(npoints, sim_len)
    for v in RECORD_VARS:
        if v == "PrecPhase":
            pa.PrecPhase[:] = fields[v]
        else:
            getattr(pa, v)[:] = fields[v]
    if analysis_hours > 0 and rec.obs_bias is not None:
        # observed atmosphere differs from the forecast one during the analysis: a jump that the
        # relaxation phase has to smooth (src/Relaxation.f90)
        n_obs = forecast_step + 1
        pa.tair[:, :n_obs] += rec.obs_bias[:, [0]]
        pa.VZ[:, :n_obs] = np.clip(pa.VZ[:, :n_obs] + rec.obs_bias[:, [1]], 0.0, 25.0)
        pa.Rhz[:, :n_obs] = np.clip(pa.Rhz[:, :n_obs] + rec.obs_bias[:, [2]], 35.0, 100.0)
        pa.TSurfObs[:, n_obs:] = -9999.9
    pa.local_horizons[:] = rec.horizons
    pa.time[:] = time_axis(sim_start, sim_len, dt)
    settings = abi.default_settings(sim_len, use_coupling, use_relaxation, dt, nlayers, **settings_kw)
    params = abi.default_parameters(dt)
    for p in range(npoints):
        lp = pa.local[p]
        lp.tair_relax = lp.VZ_relax = lp.RH_relax = -9999.0
        lp.couplingIndexI = -9999
        lp.couplingTsurf = -9999.0
        lp.lat, lp.lon, lp.sky_view = rec.lat[p], rec.lon[p], rec.sky_view[p]
        lp.InitLenI = 0
    read_input_derive(pa, settings, forecast_step)
    return pa, settings, params


def make_case(npoints, hours, seed, analysis_hours=0, use_coupling=0, use_relaxation=0,
              dt=30.0, nlayers=15, start=None, sky_view_fraction=0.3, obs_bias=True, settings_kw=None,
              **kw):
    """Seeded full-resolution host-layout case: (PointArrays, InputSettings, InputParameters, Records).

    The simulation starts `analysis_hours` before `start` (default FORECAST_START) and runs
    `hours` of forecast: SimLen = 1 + (analysis_hours + hours) * 3600 / dt."""
    start = start or FORECAST_START
    sim_start = start - _dt.timedelta(hours=analysis_hours)
    nrec = analysis_hours + hours + 2
    rec = draw_records(npoints, nrec, seed, sim_start, 3600, dt, 0, sky_view_fraction, **kw)
    if analysis_hours > 0:
        # observations exist up to forecast start; none afterwards
        rec.TSurfObs[:, analysis_hours + 1:] = -9999.9
        if obs_bias:
            rng = np.random.Generator(np.random.PCG64(seed + 77))
            rec.obs_bias = np.stack([rng.normal(0.0, 1.0, npoints), rng.normal(0.0, 0.7, npoints),
                                     rng.normal(0.0, 4.0, npoints)], axis=1)
    else:
        rec.TSurfObs[:, :] = -9999.9
    pa, settings, params = case_from_records(rec, hours, analysis_hours, use_coupling, use_relaxation, dt,
                                             nlayers, start, **(settings_kw or {}))
    return pa, settings, params, rec


def member_records(base, members, r_f, seed, start, dt_secs=30.0, sky_view_fraction=0.3):
    """`members` record sets of an ensemble forked after record r_f: member m equals `base` (drawn by
    draw_records with the same seed, start, spacing and sky-view fraction) in every record up to r_f and
    in its observations, and is a perturbed draw (draw_records(..., member_perturbation=m)) after r_f.
    Each is a full record set: it is what an independent run of member m reads."""
    record_secs = float(base.record_step[1] - base.record_step[0]) * dt_secs
    out = []
    for m in range(members):
        r = draw_records(base.npoints, base.nrec, seed, start, record_secs, dt_secs, int(base.record_step[0]),
                         sky_view_fraction, member_perturbation=m)
        for v in RECORD_VARS:
            getattr(r, v)[:, :r_f + 1] = getattr(base, v)[:, :r_f + 1]
        r.TSurfObs[:] = base.TSurfObs
        r.lat[:], r.lon[:], r.sky_view[:], r.horizons[:] = base.lat, base.lon, base.sky_view, base.horizons
        r.record_step[:] = base.record_step
        r.obs_bias = None
        out.append(r)
    return out


def member_record_tensor(member_recs, r_f):
    """The members' records r_f + 1 ... as [n_records - r_f - 1][11][P * M] (lane p * M + m), the layout of
    roadsurf_run_ensemble_host_soa's member_records."""
    M, P, nrec = len(member_recs), member_recs[0].npoints, member_recs[0].nrec
    out = np.zeros((nrec - r_f - 1, len(RECORD_VARS), P * M))
    for m, r in enumerate(member_recs):
        for v, name in enumerate(RECORD_VARS):
            out[:, v, m::M] = getattr(r, name)[:, r_f + 1:].T
    return out


def lane_records(member_recs):
    """One Records object whose point p * M + m is member m of station p: the input of P * M independent
    runs."""
    M, P, nrec = len(member_recs), member_recs[0].npoints, member_recs[0].nrec
    r = Records(P * M, nrec)
    for v in RECORD_VARS:
        a = getattr(r, v)
        for m, mr in enumerate(member_recs):
            a[m::M] = getattr(mr, v)
    for m, mr in enumerate(member_recs):
        r.lat[m::M], r.lon[m::M], r.sky_view[m::M], r.horizons[m::M] = mr.lat, mr.lon, mr.sky_view, mr.horizons
    r.record_step[:] = member_recs[0].record_step
    return r
