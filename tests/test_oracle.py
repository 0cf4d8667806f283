"""Pins the CPU oracle: against the golden vectors the UNMODIFIED reference produced
(oracle/make_golden.py), against the installed SciPy / NumPy routines the reference
calls, and -- in the build container only -- against the reference run live."""
import os

import numpy as np
import pytest

from oracle import mica_oracle as orc
from oracle import ref_harness as rh
from mica_b200 import synthetic

from _golden import load_stitch


def test_normalize_and_encode_match_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, 'preprocess_small.npz'))
    res = orc.resample(g['src'], g['voxel'])
    assert np.array_equal(res, g['oracle_resampled'])
    norm, med, p = orc.normalize(res)
    assert np.array_equal(norm, g['ref_normalized'])                # reference output, bit for bit
    assert np.float32(med) == g['median'] and np.float32(p) == g['p999']
    vol, ok = orc.af3_encode(g['coords'], g['bb_ch'], g['aa_ch'], g['origin'], norm.shape)
    assert ok == bool(g['af3_ok'])                                  # non-cubic grid: IndexError path (D7)
    g = np.load(os.path.join(golden_dir, 'af3_cubic.npz'))
    vol, ok = orc.af3_encode(g['coords'], g['bb_ch'], g['aa_ch'], g['origin'], tuple(g['shape']))
    assert ok and np.array_equal(np.argwhere(vol > 0).astype(np.int32), g['af3_nonzero'])


def test_cubes_match_reference_golden(golden_dir):
    g = np.load(os.path.join(golden_dir, 'cubes.npz'))
    vol = np.random.default_rng(2022).random((50, 100, 70), dtype=np.float32)
    cubes, meta, shp, off = orc.extract_cubes(vol, nstart_zyx=(11, -7, 4))
    assert shp == (70, 100, 50) and np.array_equal(meta, g['d_meta']) and list(off) == list(g['d_offset'])
    assert np.array_equal([np.bitwise_xor.reduce(c.view(np.uint32).ravel()) for c in cubes], g['d_xor'])
    c2, m2, _, _ = orc.extract_cubes(g['s_vol'], grid_size=8, padding=2)
    assert np.array_equal(c2, g['s_cubes']) and np.array_equal(m2, g['s_meta'])
    c3, m3, _, o3 = orc.extract_cubes(g['s_vol'], 2, 3, 1, (3, 2, 1), 8, 2)
    assert np.array_equal(c3, g['a_cubes']) and np.array_equal(m3, g['a_meta']) and list(o3) == list(g['a_offset'])
    c4, m4, _, _ = orc.extract_cubes(g['t_vol'], grid_size=8, padding=2, transpose=False, drop_below=0.01)
    assert np.array_equal(m4, g['t_meta'])


def test_stitch_matches_reference_golden(golden_dir):
    g = load_stitch(golden_dir)
    bb, ca, aa = synthetic.synthetic_logits(len(g['meta']), 64, seed=int(g['logits_seed']))
    got = orc.postprocess_and_stitch(bb, ca, aa, g['meta'], tuple(g['orig_shape']))
    for k, v in got.items():
        assert v.dtype == np.float32 and np.array_equal(v, g[k]), k


@pytest.mark.parametrize('shape,zf', [((20, 23, 17), (1.06, 1.06, 1.06)), ((30, 30, 30), (0.83, 1.31, 1.0)),
                                      ((30, 12, 9), (1.2, 1.2, 1.2)), ((5, 4, 3), (2.0, 2.5, 3.0))])
@pytest.mark.parametrize('order', [3, 1])
def test_restated_zoom_equals_scipy(shape, zf, order):
    from scipy.ndimage import zoom
    x = np.random.default_rng(1).normal(size=shape).astype(np.float32)
    zf = [np.float32(z) for z in zf]
    want = zoom(x, zf, order=order)
    got = orc.resample_restated(x, zf, order=order)
    assert got.shape == want.shape
    # SciPy zeroes output planes whose coordinate overshoots n-1 by rounding (D11); compare elsewhere
    mask = np.ones(want.shape, bool)
    for a in range(3):
        n_in, n_out = shape[a], want.shape[a]
        if n_out > 1 and (n_out - 1) * ((n_in - 1) / (n_out - 1)) > n_in - 1:
            idx = [slice(None)] * 3
            idx[a] = n_out - 1
            assert not want[tuple(idx)].any()
            mask[tuple(idx)] = False
    assert np.abs(got - want)[mask].max() <= 1e-6 * np.abs(want).max()


def test_identity_zoom_is_a_copy():
    x = np.random.default_rng(2).normal(size=(7, 8, 9)).astype(np.float32)
    assert np.array_equal(orc.resample(x, (1.0, 1.0, 1.0)), x)          # D10
    assert np.array_equal(orc.resample_restated(x, [np.float32(1)] * 3), x)


@pytest.mark.parametrize('n', [1, 2, 5, 1000, 1001, 65537, (1 << 24) + 77])
def test_order_stats_recipe_equals_numpy(n):
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n, dtype=np.float32)
    med, p, npos = orc.order_stats_restated(x)
    assert med == np.median(x)
    m = (x > np.median(x)) * (x - np.median(x))
    pos = m[m > 0]
    assert npos == len(pos)
    if npos:
        assert p == np.percentile(pos, 99.9)


def test_af3_rounding_is_half_even_and_clip_is_quirky():
    origin = (np.float32(0), np.float32(0), np.float32(0))
    c = np.array([[2.5, 3.5, 0.5], [-0.5, 1.5, 4.49]], np.float32)
    vol, ok = orc.af3_encode(c, np.array([0, 1], np.int8), np.array([-1, -1], np.int8), origin, (8, 8, 8))
    assert ok and vol[0, 0, 4, 2] == 1 and vol[1, 4, 2, 0] == 1 and vol.sum() == 2
    idx = orc.transform_coordinates(np.array([65.2, 10, 20], np.float32),
                                    np.rec.array((0., 0., 0.), dtype=[('x', 'f4'), ('y', 'f4'), ('z', 'f4')]).tolist(),
                                    (50, 100, 70))
    assert list(idx) == [49, 10, 20]                                    # x clamped by nz - 1 (D7)


@pytest.mark.skipif(not rh.available(), reason='/root/reference only exists in the build container')
def test_oracle_against_live_reference(tmp_path):
    src = synthetic.synthetic_map((18, 20, 16), seed=21)
    voxel = (np.float32(1.1), np.float32(1.1), np.float32(1.1))
    norm, path, dp = rh.resample_and_normalize(src, voxel, str(tmp_path))
    o_norm, _, _ = orc.normalize(orc.resample(src, voxel))
    assert np.array_equal(norm, o_norm)
    n, offset, cubes, shp = rh.grids_from_mrc(path, str(tmp_path / 'g'), 8, 3)
    oc, om, oshp, _ = orc.extract_cubes(o_norm, grid_size=8, padding=3)
    assert n == len(oc) and shp == tuple(oshp)
    for c, m in zip(oc, om):
        assert np.array_equal(cubes[tuple(m[:3])][0], c)


def test_training_twins_match_reference_golden(golden_dir, tmp_path):
    """scripts_for_training_data/create_normalized_map.py + create_AF3_encodings.py outputs
    (produced by the unmodified reference, oracle/make_golden.py::golden_training_twins)."""
    from mica_b200.pdb import read_pdb_atoms
    g = np.load(os.path.join(golden_dir, 'training_twins.npz'))
    norm, _, _ = orc.normalize(orc.resample(g['src'], g['voxel']))
    assert np.array_equal(norm, g['normalized'])
    pdb_path = tmp_path / 'x_af3_docked.pdb'
    pdb_path.write_text(str(g['pdb_text']))
    coords, bb, aa, _ = read_pdb_atoms(str(pdb_path))
    vol, ok = orc.af3_encode(coords, bb, aa, g['origin'], g['enc_map'].shape)
    assert ok and np.array_equal(np.argwhere(vol > 0).astype(np.int32), g['enc_nonzero'])


def test_streamed_whole_path_equals_front_plus_stitch():
    """bench.py's CPU arm (chunked, bounded memory) is the same arithmetic as the one-shot functions."""
    src = synthetic.synthetic_map((20, 24, 18), voxel=1.2, seed=3)
    voxel = (np.float32(1.2),) * 3
    n_out = orc.zoom_output_shape(src.shape, orc.zoom_factors(voxel))
    st = synthetic.synthetic_structure(30, n_out[::-1], seed=3)
    bb_ch, aa_ch = orc.channel_codes(st['atom_names'], st['res_names'])
    norm, af3, x, af, meta, shp, _ = orc.pipeline_front(src, voxel, st['coords'], bb_ch, aa_ch, (0, 0, 0), 16, 8)
    ring = synthetic.synthetic_logits(len(meta), 32, seed=1)
    want = orc.postprocess_and_stitch(*ring, meta, shp, 8)
    for chunk in (len(meta), 3):
        r = tuple(t[:chunk] for t in ring)
        if chunk < len(meta):       # the ring is reused per chunk: build the matching one-shot logits
            idx = np.arange(len(meta)) % chunk
            want = orc.postprocess_and_stitch(*(t[idx] for t in r), meta, shp, 8)
        vols, nvox, ncubes = orc.pipeline_whole_streamed(src, voxel, st['coords'], bb_ch, aa_ch, (0, 0, 0), r, 16, 8)
        assert nvox == norm.size and ncubes == len(meta)
        for k in want:
            assert np.array_equal(vols[k], want[k]), k
