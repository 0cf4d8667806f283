"""Integer maps (int8 / int16 / uint16, MRC modes 0, 1, 6; DESIGN.md D12) on the GPU: the rounded resample
against scipy.ndimage.zoom on the integer array through every kernel each type reaches, the float64 order
statistics against np.median / np.percentile, the normalised volume bit for bit against the oracle, and the
drop-in sequence on integer map files."""
import logging
import os

import numpy as np
import pytest
import torch
from scipy.ndimage import zoom

from mica_b200 import _lib, mrc, ops, pdb, session, synthetic
from mica_b200.create_grids import GridCreator
from mica_b200.pipeline import MapHeader, MapPipeline
from mica_b200.predict import CryoEMPredictor
from mica_b200.preprocessing import DataPreprocessor, upload_map
from mica_b200.slab import SlabPipeline
from oracle import mica_oracle as orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT_TYPES = (np.int8, np.int16, np.uint16)
TORCH = {np.int8: torch.int8, np.int16: torch.int16, np.uint16: torch.uint16}


def _rs_ids():
    import re
    text = open(os.path.join(ROOT, 'include', 'mica_b200.h')).read()
    return {int(v): name for name, v in re.findall(r'#define MICA_RS_(\w+) (\d+)', text)}


RS_NAME = _rs_ids()


def route():
    return tuple(RS_NAME.get(_lib.lib.mica_last_resample_path(p)) for p in range(4))


def _to_dev(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _to_host(t):
    return t.cpu().numpy()


def _inputs(dtype, shape, seed):
    """Full-range noise (the cubic spline overshoots: saturating stores) and a density-like map scaled to the
    type's range (smooth, mostly background)."""
    info = np.iinfo(dtype)
    rng = np.random.default_rng(seed)
    noise = rng.integers(int(info.min), int(info.max) + 1, shape).astype(dtype)
    d = synthetic.synthetic_map(shape, seed=seed)
    d = (d - d.min()) / max(float(d.max() - d.min()), 1e-6)
    smooth = np.round(info.min + d.astype(np.float64) * (float(info.max) - info.min) * 0.9).astype(dtype)
    return noise, smooth


def _compare_with_scipy(got, a, zf, order):
    """got must equal zoom(a) except where SciPy's float64 value lies within 1e-9 of a k + 1/2 boundary."""
    want = zoom(a, zf, order=order)
    assert got.shape == want.shape and got.dtype == want.dtype
    diff = got != want
    n_diff = int(diff.sum())
    if n_diff:
        f64 = zoom(a.astype(np.float64), zf, order=order)
        near = np.abs(np.abs(f64) - np.floor(np.abs(f64)) - 0.5) < 1e-9
        assert not (diff & ~near).any(), f'{int((diff & ~near).sum())} voxels differ away from a rounding boundary'
        assert (np.abs(got.astype(np.int64) - want.astype(np.int64))[diff] <= 1).all()
    print(f'{a.dtype} {a.shape} -> {want.shape}: {n_diff} voxels at a k + 1/2 boundary differ')
    return n_diff


# (id, source shape, zoom factors (z, y, x), order, expected z prefilter, expected interpolation kernel)
CASES = [
    ('seg16_tma3', (100, 30, 32), (1.2, 1.2, 1.2), 3, 'COLS_SEG16', 'MARCH3_TMA3'),
    ('cols32_tma4', (40, 42, 44), (0.8, 0.8, 0.8), 3, 'COLS32', 'MARCH3_TMA4'),
    ('cols8_march3', (900, 9, 11), (1.1, 1.1, 1.1), 3, 'COLS8', 'MARCH3_3'),
    ('global_march4', (3300, 6, 7), (0.8, 0.8, 0.8), 3, 'COLS_GLOBAL', 'MARCH3_4'),
    ('gather3', (20, 3, 24), (1.3, 1.3, 1.3), 3, 'COLS32', 'GATHER3'),
    ('gather1', (30, 31, 33), (1.2, 1.2, 1.2), 1, None, 'GATHER1'),
    ('anisotropic', (50, 52, 54), (1.1, 0.9, 1.3), 3, 'COLS32', None),
    ('d11_30_to_36', (30, 30, 30), (1.2, 1.2, 1.2), 3, 'COLS32', 'MARCH3_TMA3'),
]


@pytest.mark.parametrize('dtype', INT_TYPES, ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize('case', CASES, ids=[c[0] for c in CASES])
def test_int_resample_equals_scipy_on_every_route(cuda, dtype, case):
    name, shape, zf, order, z_kernel, interp = case
    zf = [np.float32(v) for v in zf]
    out_shape = ops.zoom_output_shape(shape, zf)
    for a in _inputs(dtype, shape, seed=len(name)):
        got = ops.resample(_to_dev(a, cuda), out_shape, order=order)
        torch.cuda.synchronize()
        assert got.dtype == TORCH[dtype]
        r = route()
        assert r[0] == z_kernel and (interp is None or r[3] == interp), r
        _compare_with_scipy(_to_host(got), a, zf, order)
    if name == 'd11_30_to_36':
        assert np.all(_to_host(got)[-1] == 0)           # the zero last plane of D11


def test_float32_resample_keeps_its_entry_point(cuda):
    a = synthetic.synthetic_map((40, 42, 44), seed=3)
    zf = [np.float32(1.2)] * 3
    out_shape = ops.zoom_output_shape(a.shape, zf)
    got = _to_host(ops.resample(_to_dev(a, cuda), out_shape))
    r1 = route()
    src = _to_dev(a, cuda)
    out = torch.empty(out_shape, dtype=torch.float32, device=cuda)
    nb = _lib.lib.mica_resample_workspace_bytes(*a.shape, *out_shape, 3)
    ws = torch.empty(nb, dtype=torch.uint8, device=cuda)
    assert _lib.lib.mica_bspline_resample_f32(src.data_ptr(), *a.shape, 0, a.shape[0], out.data_ptr(), *out_shape, 0,
                                              out_shape[0], ws.data_ptr(), nb, 3,
                                              torch.cuda.current_stream().cuda_stream) == 0
    assert route() == r1
    assert np.array_equal(_to_host(out).view(np.uint32), got.view(np.uint32))
    with pytest.raises(_lib.MicaError):
        ops.resample(_to_dev(a, cuda), out_shape, out=torch.empty(out_shape, dtype=torch.int16, device=cuda))


# -------------------------------------------------------------- statistics and normalise
def _check_stats(x, dev):
    """IntOrderStats + apply on x against NumPy's float64 statistics and the oracle's normalisation."""
    xd = _to_dev(x, dev)
    st = ops.IntOrderStats(dev).run(xd)
    med, p, npos, status = st.result()
    assert isinstance(med, float) and isinstance(p, float)
    want_med = np.median(x)
    assert med == want_med, (med, want_med)
    want, _, want_p = orc.normalize(x)
    m = (x > want_med) * (x - want_med)
    assert npos == int((m > 0).sum())
    rec = st.result_async()
    torch.cuda.synchronize()
    assert ops.IntOrderStats.decode(rec) == (med, p, npos, status)
    if want is None:
        assert status == (_lib.NORM_NO_POSITIVE if npos == 0 else _lib.NORM_ZERO_PCTL)
        return status
    assert status == _lib.NORM_OK and p == want_p, (p, want_p)
    got = _to_host(st.apply(xd))
    assert got.dtype == np.float32 and np.array_equal(got.view(np.uint32), want.view(np.uint32))
    norm, _ = ops.normalize(xd)
    assert np.array_equal(_to_host(norm).view(np.uint32), want.view(np.uint32))
    with pytest.raises(_lib.MicaError):
        ops.normalize(xd, inplace=True)
    return status


def test_int_stats_on_hand_built_volumes(cuda):
    rng = np.random.default_rng(11)
    cases = [
        np.array([[[5]]], dtype=np.int16),                                      # n = 1: no positives
        np.array([1, 2, 3, 4, 10, 20, 30, 40], dtype=np.int8).reshape(2, 2, 2),  # even n, half-integer median
        np.arange(27, dtype=np.uint16).reshape(3, 3, 3),                         # odd n
        rng.integers(-5, 6, (4, 5, 6)).astype(np.int16),                         # even n, ties
        rng.integers(-5, 6, (3, 5, 7)).astype(np.int16),                         # odd n, ties
        np.full((6, 7, 8), -3, dtype=np.int8),                                   # all equal: no positives
        np.tile(np.arange(-128, 128, dtype=np.int8), 64).reshape(16, 32, 32),   # full-range int8
        rng.integers(0, 65536, (64, 64, 64)).astype(np.uint16),                  # full-range uint16
        rng.integers(-128, 128, (33, 35, 37)).astype(np.int8),
    ]
    x = np.zeros((4, 4, 4), dtype=np.uint16)
    x[0, 0, 0], x[1, 1, 1] = 7, 9                                               # npos = 2
    cases.append(x)
    statuses = [_check_stats(c, cuda) for c in cases]
    assert statuses[0] == _lib.NORM_NO_POSITIVE and statuses[5] == _lib.NORM_NO_POSITIVE
    assert statuses.count(_lib.NORM_OK) == len(cases) - 2


@pytest.mark.parametrize('dtype', INT_TYPES, ids=lambda d: np.dtype(d).name)
def test_int_stats_on_gpu_resampled_maps(cuda, dtype):
    for a in _inputs(dtype, (60, 62, 64), seed=4):
        zf = [np.float32(1.1)] * 3
        res = ops.resample(_to_dev(a, cuda), ops.zoom_output_shape(a.shape, zf))
        assert _check_stats(_to_host(res), cuda) == _lib.NORM_OK


def test_int16_stats_at_480_cubed(cuda):
    rng = np.random.default_rng(12)
    d = synthetic.synthetic_map_device((480, 480, 480), cuda, voxel=1.0, seed=12)
    d = (d - d.min()) / (d.max() - d.min())
    x = torch.round(d.double() * 60000 - 30000).to(torch.int16)
    x[:4].copy_(torch.from_numpy(rng.integers(-32768, 32768, (4, 480, 480)).astype(np.int16)))
    del d
    xh = _to_host(x)
    st = ops.IntOrderStats(cuda).run(x)
    med, p, npos, status = st.result()
    want, want_med, want_p = orc.normalize(xh)
    assert status == _lib.NORM_OK and med == want_med and p == want_p
    got = _to_host(st.apply(x))
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_pipeline_on_integer_sources(cuda):
    pipe = MapPipeline(cuda, grid_size=32, padding=8, batch_cubes=4)
    for dtype in INT_TYPES:
        noise, smooth = _inputs(dtype, (40, 44, 36), seed=9)
        for voxel in (1.2, 1.0):                                          # 1.0: the D10 copy
            hdr = MapHeader(voxel_size=(np.float32(voxel),) * 3)
            src = _to_dev(smooth, cuda)
            assert pipe.resample_and_normalize(src, hdr)
            want, med, p = orc.normalize(orc.resample(smooth, hdr.voxel_size))
            assert pipe.normalized.dtype == torch.float32
            assert np.array_equal(_to_host(pipe.normalized).view(np.uint32), want.view(np.uint32))
            assert isinstance(pipe.median, float) and pipe.median == med and pipe.p999 == p
            assert np.array_equal(_to_host(src), smooth)                  # the source is not overwritten
            assert pipe.resample_and_normalize(src, hdr, defer_status=True) and pipe.check_status()
    flat = torch.full((20, 20, 20), 3, dtype=torch.int16, device=cuda)
    assert not pipe.resample_and_normalize(flat, MapHeader(voxel_size=(np.float32(1.2),) * 3))
    assert pipe.normalized is None and pipe.norm_status == _lib.NORM_NO_POSITIVE


def test_upload_keeps_the_integer_type(cuda):
    for dtype in INT_TYPES:
        a = np.random.default_rng(2).integers(0, 100, (128, 128, 300)).astype(dtype)    # > 2^22: staged path
        t = upload_map(a, cuda)
        assert t.dtype == TORCH[dtype] and np.array_equal(_to_host(t), a)
    f = np.random.default_rng(2).standard_normal((128, 128, 300)).astype(np.float32)
    assert np.array_equal(_to_host(upload_map(f, cuda)), f)


def test_slab_pipeline_refuses_integer_maps(cuda):
    p = SlabPipeline(cuda, 0, 1, 48, 8, global_src_shape=(40, 40, 40), group=False)
    with pytest.raises(_lib.MicaError, match='int16'):
        p.resample_and_normalize(torch.zeros((40, 40, 40), dtype=torch.int16, device=cuda),
                                 MapHeader(voxel_size=(np.float32(1.2),) * 3))


# ------------------------------------------------------------------------ drop-in
class PointwiseModel(torch.nn.Module):
    """The stand-in of tests/test_gpu_dropin.py: elementwise, so the oracle can evaluate it on its cubes."""

    def forward(self, x, af):
        s = af.sum(dim=1, keepdim=True)
        bb = torch.cat([x, -x, 2 * x - 0.5 + s, x * x], dim=1)
        ca = torch.cat([0.5 - x, x, x * 3 - 1, 1.5 * x + af[:, :1]], dim=1)
        aa = torch.cat([x * (0.1 * t) + af[:, t % 24:t % 24 + 1] * (t % 3) + np.sin(t) for t in range(21)], dim=1)
        return bb, ca, aa


def _write_case(tmp_path, data, voxel, tag, dtype=None):
    case = tmp_path / tag / 'input' / 'ID'
    os.makedirs(case / 'AF3_results', exist_ok=True)
    origin = (np.float32(12.5), np.float32(-4.0), np.float32(0.75))
    map_path = str(case / 'map.mrc')
    mrc.write_mrc(map_path, mrc.MrcMap(data=data, voxel_size=(np.float32(voxel),) * 3, origin=origin, nxstart=2,
                                       nystart=3, nzstart=5), dtype=dtype or data.dtype)
    n = round(data.shape[0] * voxel)
    st = synthetic.synthetic_structure(150, (n, n, n), seed=31, origin_xyz=origin, hetero_every=13)
    pdb_path = str(case / 'ID_af3_docked.pdb')
    synthetic.write_pdb(pdb_path, st)
    return origin, map_path, pdb_path, str(case / 'AF3_results'), str(case / 'grids')


@pytest.mark.parametrize('dtype,shape', [(np.int16, (40, 40, 40)), (np.int8, (24, 24, 24)),
                                         (np.uint16, (24, 24, 24))], ids=['int16', 'int8', 'uint16'])
def test_dropin_sequence_on_integer_map_files(cuda, tmp_path, dtype, shape):
    session.clear()
    voxel = 1.1
    src = _inputs(dtype, shape, seed=31)[1]
    origin, map_path, pdb_path, af3_results, grids_path = _write_case(tmp_path, src, voxel, 'a')
    assert mrc.read_mrc(map_path).mode == {np.int8: 0, np.int16: 1, np.uint16: 6}[dtype]
    dp = DataPreprocessor(map_path=map_path, AF3_results=af3_results, quiet=True, write_files=True)
    assert dp.resample_and_normalize_map() is None
    o_norm, _, _ = orc.normalize(orc.resample(src, (np.float32(voxel),) * 3))
    written = mrc.read_mrc(dp.normalized_map_path)
    assert written.mode == 2 and np.array_equal(written.data.view(np.uint32), o_norm.view(np.uint32))
    assert dp.create_AF3_encodings(pdb_path) is True
    coords, bb_ch, aa_ch, _ = pdb.read_pdb_atoms(pdb_path)
    o_af3, ok = orc.af3_encode(coords, bb_ch, aa_ch, origin, o_norm.shape)
    assert ok
    gc = GridCreator(quiet=True)
    r1 = gc.create_normalized_map_grids(dp.normalized_map_path, os.path.join(grids_path, 'normalized_map_grids'))
    r2 = gc.create_AF3_encodings_grids(dp.AF3_encodings, os.path.join(grids_path, 'AF3_encoding_grids'))
    o_cubes, o_meta, o_shape, o_off = orc.extract_cubes(o_norm, nstart_zyx=(5, 3, 2))
    assert r1['success'] and r1['grid_count'] == len(o_cubes) and r1['offset'] == o_off
    assert r2['success'] and r2['successful_channels'] == 24
    pr = CryoEMPredictor(model_path='unused', grids_path=grids_path, output_path=str(tmp_path / 'out'),
                         save_output=False, device='cuda', quiet=True, model=PointwiseModel())
    ok, vols = pr.run_prediction()
    assert ok
    vols = {k: np.asarray(v) for k, v in vols.items()}
    o_x = torch.from_numpy(orc.extract_cubes(o_norm)[0][:, None])
    o_af = torch.from_numpy(np.stack([orc.extract_cubes(o_af3[c])[0] for c in range(24)], axis=1))
    with torch.no_grad():
        bb, ca, aa = PointwiseModel()(o_x, o_af)
    want = orc.postprocess_and_stitch(bb, ca, aa, o_meta, o_shape)
    for k in ('backbone_probability', 'carbon_alpha_probability', 'amino_acid_probability'):
        assert vols[k].shape == want[k].shape and np.abs(vols[k] - want[k]).max() <= 2e-5, k
    top2 = np.sort(want['amino_acid_probability'], axis=0)[-2:]
    clear = (top2[1] - top2[0]) > 4e-6
    assert np.array_equal(vols['amino_acid_prediction'][clear], want['amino_acid_prediction'][clear])


def test_dropin_flat_integer_map_and_float16_refusal(cuda, tmp_path, caplog):
    session.clear()
    flat = np.full((20, 20, 20), 12, dtype=np.int16)
    _, map_path, _, af3_results, _ = _write_case(tmp_path, flat, 1.1, 'flat')
    dp = DataPreprocessor(map_path=map_path, AF3_results=af3_results, quiet=True)
    with caplog.at_level(logging.ERROR):
        dp.resample_and_normalize_map()
    assert dp.normalized_map_path is None and 'No positive values' in caplog.text
    caplog.clear()
    half = np.random.default_rng(1).standard_normal((20, 20, 20)).astype(np.float16)
    _, map_path, _, af3_results, _ = _write_case(tmp_path, half, 1.1, 'half')
    assert mrc.read_mrc(map_path).mode == 12
    dp = DataPreprocessor(map_path=map_path, AF3_results=af3_results, quiet=True)
    with caplog.at_level(logging.ERROR):
        dp.resample_and_normalize_map()
    assert dp.normalized_map_path is None and 'mode 12' in caplog.text
