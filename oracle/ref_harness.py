"""TEST INFRASTRUCTURE -- runs the UNMODIFIED reference (tepextepex/ENRGY) under stub modules.

Only usable where the reference checkout exists (this container: /root/reference). It is used by
`tests/golden/make_golden.py` to generate the committed golden fixtures and by the `not gpu` tests
that pin `oracle/enrgy_oracle.py` against the real reference. Nothing on the GPU box imports it
(/root/reference does not exist there), and nothing in the product package `enrgy_b200/` may import
anything from `oracle/`.

How the reference is made runnable without GDAL / matplotlib / SAGA (SURVEY.md section 8c):
  1. fake `osgeo`, `osgeo.gdal`, `matplotlib`, `matplotlib.pyplot` are put into sys.modules;
  2. `model.load_raster`, `model.show_me`, `model.export_array_as_geotiff` (imported by name at
     reference model.py:10) are rebound to array-backed versions;
  3. insolation is fed through the reference's own cache path: `use_precomputed = True`,
     `add_pickle_dir(dir)`, files `<dir>/<res>/<DATE>_total.sdat.npy` (model.py:465-481);
  4. `model.OutputRow` and `model.calc_melt` are wrapped by recorders so the per-step flux rasters
     can be captured -- the wrapped callables are the reference's own objects, untouched.
"""
from __future__ import annotations

import importlib
import io
import os
import sys
import tempfile
import types
import contextlib

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _find_reference():
    """ENRGY_REFERENCE_DIR, else the declared reference checkout (BASELINE.json reference_path), else
    the unmodified copy __graft_entry__.build() puts under oracle/_ref/ (git-ignored)."""
    for d in (os.environ.get("ENRGY_REFERENCE_DIR"), "/root/reference", os.path.join(_ROOT, "oracle", "_ref")):
        if d and os.path.isfile(os.path.join(d, "model.py")):
            return d
    return os.environ.get("ENRGY_REFERENCE_DIR", "/root/reference")


REFERENCE_DIR = _find_reference()


def reference_available():
    return os.path.isfile(os.path.join(REFERENCE_DIR, "model.py"))


def _install_stubs():
    if "osgeo" not in sys.modules:
        osgeo = types.ModuleType("osgeo")
        gdal = types.ModuleType("osgeo.gdal")
        gdal.GDT_Float32 = 6
        gdal.GDT_Int16 = 3
        osgeo.gdal = gdal
        sys.modules["osgeo"] = osgeo
        sys.modules["osgeo.gdal"] = gdal
    if "matplotlib" not in sys.modules:
        mpl = types.ModuleType("matplotlib")
        plt = types.ModuleType("matplotlib.pyplot")
        for name in ("imshow", "title", "colorbar", "savefig", "show", "clf", "subplots"):
            setattr(plt, name, lambda *a, **k: None)
        mpl.pyplot = plt
        sys.modules["matplotlib"] = mpl
        sys.modules["matplotlib.pyplot"] = plt


def import_reference():
    """Returns the reference's modules as a namespace (model, turbo, msm, helpers, ...)."""
    if not reference_available():
        raise RuntimeError("reference checkout not found at %s" % REFERENCE_DIR)
    _install_stubs()
    if REFERENCE_DIR not in sys.path:
        sys.path.insert(0, REFERENCE_DIR)
    ns = types.SimpleNamespace()
    for name in ("turbo", "helpers", "interpolator", "var_classes", "msm", "model", "saga_lighting",
                 "beer_lambert"):
        ns.__dict__[name] = importlib.import_module(name)
    return ns


class _Recorder:
    """Records the arrays handed to OutputRow(...) and returned by calc_melt(...) at every step."""

    def __init__(self, ref, keep_steps=None):
        self.ref = ref
        self.keep = keep_steps
        self.rows = []       # per step dict of arrays
        self.melt = []       # per step (snow, ice)
        self._orig_row = ref.model.OutputRow
        self._orig_melt = ref.model.calc_melt

    def __enter__(self):
        rec = self

        def make_row(date_time_str, lwd, lwu, rs, sens, lat, atmo, g, mf, pts):
            i = len(rec.rows)
            if rec.keep is None or i in rec.keep:
                rec.rows.append(dict(date=date_time_str, lwd=np.array(lwd), lwu=np.array(lwu),
                                     rs=np.array(rs), sens=np.array(sens), lat=np.array(lat),
                                     atmo=np.array(atmo), g=np.array(g), mf=np.array(mf),
                                     point_t_surf=float(pts)))
            else:
                rec.rows.append(None)
            return rec._orig_row(date_time_str, lwd, lwu, rs, sens, lat, atmo, g, mf, pts)

        def melt(melt_flux, swe, time_step):
            out = rec._orig_melt(melt_flux, swe, time_step)
            i = len(rec.melt)
            if rec.keep is None or i in rec.keep:
                rec.melt.append((np.array(out[0]), np.array(out[1]), np.array(swe)))
            else:
                rec.melt.append(None)
            return out

        self.ref.model.OutputRow = make_row
        self.ref.model.calc_melt = melt
        return self

    def __exit__(self, *exc):
        self.ref.model.OutputRow = self._orig_row
        self.ref.model.calc_melt = self._orig_melt


def run_reference(case, insolation, *, f64=False, const_albedo=None, use_albedo_maps=True,
                  z=1.6, zm=1e-3, z_h_or_e=1e-4, andreas=False, emissivity=0.98,
                  temp_lapse_rate=-0.006, last_snowfall=None, max_ice_albedo=None,
                  cloud_corr=None, sensible_corr=1, latent_corr=1, use_swe=True,
                  msm=None, snow_density=None, keep_steps=None, res=10, quiet=True):
    """Run reference `Energy.model` on a SyntheticCase.

    insolation: array [T, H, W] (kWh m-2 per step) or callable(step_index) -> [H, W].
    f64=False: as shipped (float32 rasters, float32 state, model.py:76-80).
    f64=True : "float64-injected" configuration of SURVEY.md 8c: the loader returns float64 arrays
               (values float32-representable), insolation float64, state arrays float64.
    msm: None or dict(depths=[...], temperatures=[...], elev=...)  (model.py:126-149).
    Returns dict(stats_csv=str, solar_csv=str, rows=[...], melt=[...], swe, total_snow, total_ice).
    """
    ref = import_reference()
    m = ref.model
    rdt = np.float64 if f64 else np.float32
    tmp = tempfile.mkdtemp(prefix="enrgy_ref_")
    out_dir = os.path.join(tmp, "out")
    pick = os.path.join(tmp, "pickle")
    os.makedirs(os.path.join(pick, str(res)))

    store = {"dem": case.dem.astype(rdt), "swe": case.swe.astype(rdt)}
    for k, a in case.albedo_maps.items():
        store["alb_" + k] = a.astype(rdt)

    def load_raster(raster_path, crop_path, res_, remove_negatives=False, remove_outliers=False, v=True):
        arr = np.array(store[raster_path], copy=True)
        if remove_outliers:             # reference raster_utils.py:48-50
            arr[arr < 0] = 0.001
            arr[arr > 1] = 1
        return arr, case.geotransform, "EPSG:32633"

    exported = {}

    def export_array_as_geotiff(arr, gt, proj, path, scale_mult=None):
        exported[os.path.basename(path)] = np.array(arr, copy=True)
        return path

    saved = (m.load_raster, m.show_me, m.export_array_as_geotiff)
    m.load_raster = load_raster
    m.show_me = lambda *a, **k: None
    m.export_array_as_geotiff = export_array_as_geotiff
    # PARAMS is a mutable module global changed by set_density (model.py:84-88): restore after.
    params_saved = dict(ref.var_classes.PARAMS)
    try:
        sink = io.StringIO() if quiet else sys.stdout
        with contextlib.redirect_stdout(sink):
            e = m.Energy("dem", "outline", out_dir, res=res)
            e.png_export = 10 ** 9
            e.use_precomputed = True
            e.add_pickle_dir(pick)
            if cloud_corr is not None:
                e.add_cloud_corr(cloud_corr)
            e.sensible_corr_factor = sensible_corr
            e.latent_corr_factor = latent_corr
            if snow_density is not None:
                e.set_density(snow=snow_density)
            if use_swe:
                e.add_snow("swe")
            if f64:
                e.swe_array = e.swe_array.astype(np.float64)
                e.total_snow_melt_array = e.total_snow_melt_array.astype(np.float64)
                e.total_ice_melt_array = e.total_ice_melt_array.astype(np.float64)
            if msm is not None:
                e.add_msm(list(msm["depths"]), list(msm["temperatures"]), msm["elev"])
            else:
                e.layer_temperatures = [np.zeros_like(e.base_dem_array)]     # SURVEY F9
            n_steps = len(case.aws_rows)
            for i, row in enumerate(case.aws_rows):
                pot = insolation(i) if callable(insolation) else insolation[i]
                np.save(os.path.join(pick, str(res), "%s_total.sdat.npy" % row["DATE"]),
                        np.asarray(pot, dtype=rdt))
            aws_csv = case.write_aws_csv(os.path.join(tmp, "aws.csv"))
            amaps = None
            if const_albedo is None and use_albedo_maps:
                amaps = {k: "alb_" + k for k in case.albedo_maps}
            import time as _time
            with _Recorder(ref, keep_steps) as rec:
                _t_model = _time.perf_counter()
                e.model(aws_file=aws_csv, albedo_maps=amaps, z=z, elev_aws=case.elev_aws,
                        xy_aws=case.xy_aws, zm=zm, z_h_or_e=z_h_or_e, andreas=andreas,
                        const_albedo=const_albedo, temp_lapse_rate=temp_lapse_rate,
                        last_snowfall=last_snowfall, max_ice_albedo=max_ice_albedo,
                        emissivity=emissivity, v=False)
                _t_model = _time.perf_counter() - _t_model
        with open(os.path.join(out_dir, "heat_fluxes.csv")) as f:
            stats_csv = f.read()
        with open(os.path.join(out_dir, "solar_output.csv")) as f:
            solar_csv = f.read()
        return dict(stats_csv=stats_csv, solar_csv=solar_csv, rows=rec.rows, melt=rec.melt,
                    swe=np.array(e.swe_array), total_snow=np.array(e.total_snow_melt_array),
                    total_ice=np.array(e.total_ice_melt_array), exported=exported,
                    layer_temperatures=None if msm is None else [np.array(t) for t in e.layer_temperatures],
                    numpy=np.__version__, n_steps=n_steps, model_seconds=_t_model)
    finally:
        m.load_raster, m.show_me, m.export_array_as_geotiff = saved
        ref.var_classes.PARAMS.clear()
        ref.var_classes.PARAMS.update(params_saved)
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
