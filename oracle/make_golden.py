"""Generates tests/golden/*.npz by running the UNMODIFIED reference here.

Run in the build container only (needs /root/reference):
    python -m oracle.make_golden
Each fixture holds the seeded inputs (or the recipe to regenerate them) and the
outputs the reference produced, so that tests on the GPU box -- where
/root/reference does not exist -- can pin both the oracle and the CUDA path.
"""
from __future__ import annotations

import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_harness as rh          # noqa: E402
from oracle import mica_oracle as orc         # noqa: E402
from oracle import candidates_oracle as cand_orc   # noqa: E402
from oracle import masks_oracle as mask_orc   # noqa: E402
from mica_b200 import synthetic               # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def _save(name, **kw):
    path = os.path.join(GOLDEN, name)
    np.savez_compressed(path, **kw)
    print(f'  wrote {name}: {os.path.getsize(path) / 1024:.0f} KiB')


def byte_planes(a):
    """float32 array -> (4,) + shape uint8, byte k of every value in plane k (deflates far better)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    return np.ascontiguousarray(np.moveaxis(a.view(np.uint8).reshape(a.shape + (4,)), -1, 0))


def golden_preprocess():
    """R1-R4: map (26,30,22) at anisotropic voxel -> normalised map + AF3 voxels."""
    rng = np.random.default_rng(2022)
    src = synthetic.synthetic_map((26, 30, 22), voxel=1.06, seed=7)
    voxel = (np.float32(1.06), np.float32(1.13), np.float32(0.97))
    origin = (np.float32(-3.25), np.float32(4.5), np.float32(1.75))
    with tempfile.TemporaryDirectory() as td:
        norm, path, dp = rh.resample_and_normalize(src, voxel, td, origin_xyz=origin,
                                                    nstart_xyz=(3, -2, 5))
        assert norm is not None
        nz, ny, nx = norm.shape
        # cubic sub-case first (no D7 quirk), then the quirky non-cubic grid
        st = synthetic.synthetic_structure(40, (nx, ny, nz), seed=11, origin_xyz=origin,
                                           margin=1.0, hetero_every=7, unknown_every=5)
        # push a few atoms outside the grid to exercise the clip
        st['coords'][::17] -= np.float32(9.0)
        pdb = os.path.join(td, 'AF3_results', 'x_af3_docked.pdb')
        synthetic.write_pdb(pdb, st)
        ok, enc = rh.af3_encodings(dp, pdb)
    res = orc.resample(src, voxel)
    o_norm, med, p = orc.normalize(res)
    assert np.array_equal(o_norm, norm), 'oracle normalise != reference'
    keep = ~st['hetero']
    bb, aa = orc.channel_codes([a for a, k in zip(st['atom_names'], keep) if k],
                               [r for r, k in zip(st['res_names'], keep) if k])
    o_enc, o_ok = orc.af3_encode(st['coords'][keep], bb, aa, origin, norm.shape)
    assert o_ok == ok, (o_ok, ok)
    if ok:
        assert np.array_equal(o_enc, enc), 'oracle AF3 encode != reference'
    _save('preprocess_small.npz', src=src, voxel=np.array(voxel), origin=np.array(origin),
          ref_normalized=norm, oracle_resampled=res, median=np.float32(med), p999=np.float32(p),
          coords=st['coords'][keep], bb_ch=bb, aa_ch=aa, af3_ok=np.bool_(ok),
          af3_nonzero=(np.argwhere(enc > 0).astype(np.int32) if ok else np.zeros((0, 4), np.int32)))


def golden_af3_cubic():
    """R4 on a cubic grid (quirk-free) incl. the reference's PDB text path."""
    with tempfile.TemporaryDirectory() as td:
        vol = np.abs(synthetic.synthetic_map((24, 24, 24), voxel=1.0, seed=3))
        origin = (np.float32(10.5), np.float32(-7.25), np.float32(0.0))
        norm, path, dp = rh.resample_and_normalize(vol, (1.0, 1.0, 1.0), td, origin_xyz=origin)
        st = synthetic.synthetic_structure(60, (24, 24, 24), seed=5, origin_xyz=origin,
                                           margin=0.5, hetero_every=9, unknown_every=4)
        st['coords'][::13] += np.float32(6.5)        # some out of range -> clipped
        # half-integer coordinates: banker's rounding (2.5 -> 2, 3.5 -> 4)
        st['coords'][1::19] = (np.floor(st['coords'][1::19] - np.array(origin, 'f')) +
                               np.float32(0.5) + np.array(origin, 'f'))
        pdb = os.path.join(td, 'AF3_results', 'x_af3_docked.pdb')
        synthetic.write_pdb(pdb, st)
        ok, enc = rh.af3_encodings(dp, pdb)
        assert ok
        from mica_b200.pdb import read_pdb_atoms
        coords, bb, aa, nres = read_pdb_atoms(pdb)
    o_enc, o_ok = orc.af3_encode(coords, bb, aa, origin, (24, 24, 24))
    assert o_ok and np.array_equal(o_enc, enc), 'oracle AF3 encode != reference (cubic)'
    _save('af3_cubic.npz', coords=coords, bb_ch=bb, aa_ch=aa, origin=np.array(origin),
          shape=np.array((24, 24, 24)), af3_nonzero=np.argwhere(enc > 0).astype(np.int32))


def golden_cubes():
    """R5: non-cubic (70,100,50) volume, reference defaults 48/8 (checksums) and a
    small-window case 8/2 stored densely; non-standard axis order; training twin."""
    rng = np.random.default_rng(2022)
    vol = rng.random((50, 100, 70), dtype=np.float32)          # (nz,ny,nx)
    out = {}
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, 'v.mrc')
        rh._write_mrc(p, vol, nstart_xyz=(4, -7, 11))
        n, offset, cubes, orig_shape = rh.grids_from_mrc(p, os.path.join(td, 'g'))
        o_cubes, o_meta, o_shape, o_off = orc.extract_cubes(vol, nstart_zyx=(11, -7, 4))
        assert n == len(o_cubes) and tuple(o_shape) == orig_shape and list(o_off) == list(offset)
        for c, m in zip(o_cubes, o_meta):
            rc, di, dj, dk = cubes[tuple(m[:3])]
            assert np.array_equal(rc, c) and (di, dj, dk) == tuple(m[3:])
        out['d_meta'] = o_meta
        out['d_offset'] = np.array(offset)
        out['d_sum'] = np.array([np.float64(c.astype(np.float64).sum()) for c in o_cubes])
        out['d_xor'] = np.array([np.bitwise_xor.reduce(c.view(np.uint32).ravel()) for c in o_cubes])
        # small window, stored densely
        small = rng.random((9, 21, 13), dtype=np.float32)
        p2 = os.path.join(td, 's.mrc')
        rh._write_mrc(p2, small)
        n2, off2, cubes2, shp2 = rh.grids_from_mrc(p2, os.path.join(td, 'g2'), 8, 2)
        o2, m2, s2, _ = orc.extract_cubes(small, grid_size=8, padding=2)
        assert n2 == len(o2)
        for c, m in zip(o2, m2):
            assert np.array_equal(cubes2[tuple(m[:3])][0], c)
        out['s_vol'], out['s_cubes'], out['s_meta'] = small, o2, m2
        # non-standard axis order (mapc,mapr,maps) = (2,3,1)
        p3 = os.path.join(td, 'a.mrc')
        rh._write_mrc(p3, small, nstart_xyz=(1, 2, 3), axes=(2, 3, 1))
        n3, off3, cubes3, shp3 = rh.grids_from_mrc(p3, os.path.join(td, 'g3'), 8, 2)
        o3, m3, s3, f3 = orc.extract_cubes(small, 2, 3, 1, (3, 2, 1), 8, 2)
        assert n3 == len(o3) and tuple(s3) == shp3 and list(f3) == list(off3)
        for c, m in zip(o3, m3):
            assert np.array_equal(cubes3[tuple(m[:3])][0], c)
        out['a_cubes'], out['a_meta'], out['a_offset'] = o3, m3, np.array(off3)
        # training twin: no transpose, drop cubes with max < 0.01
        sparse = small.copy()
        sparse[:, :12, :] *= 0.005
        p4 = os.path.join(td, 't.mrc')
        rh._write_mrc(p4, sparse)
        n4, cubes4 = rh.training_grids_from_mrc(p4, os.path.join(td, 'g4'), 8, 2)
        o4, m4, _, _ = orc.extract_cubes(sparse, grid_size=8, padding=2, transpose=False,
                                         drop_below=0.01)
        assert n4 == len(o4) == len(cubes4) and n4 < len(o2)
        for c, m in zip(o4, m4):
            assert np.array_equal(cubes4[tuple(m[:3])][0], c)
        out['t_vol'], out['t_meta'] = sparse, m4
    _save('cubes.npz', **out)


def golden_training_twins():
    """R1/R2/R4 training twins (scripts_for_training_data/create_normalized_map.py,
    create_AF3_encodings.py): same arithmetic as the inference entry points -- asserted here
    against the reference's own DataPreprocessor -- stored with the text PDB they parsed."""
    with tempfile.TemporaryDirectory() as td:
        src = synthetic.synthetic_map((22, 26, 20), voxel=1.15, seed=17)
        voxel = (np.float32(1.15),) * 3
        origin = (np.float32(-4.5), np.float32(3.25), np.float32(8.0))
        norm_tw, tw_path = rh.training_map_processor(src, voxel, td, origin_xyz=origin)
        norm_inf, _, _ = rh.resample_and_normalize(src, voxel, os.path.join(td, 'inf'), origin_xyz=origin)
        assert norm_tw is not None and np.array_equal(norm_tw, norm_inf), 'training twin != inference path'
        o_norm, _, _ = orc.normalize(orc.resample(src, voxel))
        assert np.array_equal(o_norm, norm_tw), 'oracle != MapProcessor'
        # cubic working grid for the encoder (the clip quirk is exercised by preprocess_small)
        cube = np.abs(synthetic.synthetic_map((20, 20, 20), voxel=1.0, seed=4))
        norm_c, c_path = rh.training_map_processor(cube, (1.0, 1.0, 1.0), os.path.join(td), origin_xyz=origin)
        st = synthetic.synthetic_structure(40, (20, 20, 20), seed=9, origin_xyz=origin, margin=0.5,
                                           hetero_every=7, unknown_every=5)
        pdb_path = os.path.join(td, 'x_af3_docked.pdb')
        synthetic.write_pdb(pdb_path, st)
        enc, names = rh.training_features_encoder(c_path, pdb_path)
        from mica_b200.pdb import CHANNEL_NAMES, read_pdb_atoms
        assert list(names) == list(CHANNEL_NAMES)
        coords, bb, aa, _ = read_pdb_atoms(pdb_path)
        o_enc, ok = orc.af3_encode(coords, bb, aa, origin, (20, 20, 20))
        assert ok and np.array_equal(o_enc, enc), 'oracle != FeaturesEncoder'
        pdb_text = open(pdb_path).read()
    _save('training_twins.npz', src=src, voxel=np.array(voxel), origin=np.array(origin), normalized=norm_tw,
          enc_map=norm_c, enc_nonzero=np.argwhere(enc > 0).astype(np.int32), pdb_text=np.array(pdb_text))


def golden_stitch():
    """R6-R8: (52,20,12)-voxel map -> 2 cubes -> replayed logits -> 4 volumes,
    through CryoEMTestDataset + run_inference + reconstruct_volume on CPU."""
    rng = np.random.default_rng(2022)
    vol = rng.random((12, 20, 52), dtype=np.float32)           # (nz,ny,nx) -> T shape (52,20,12)
    enc = (rng.random((24, 12, 20, 52)) < 0.01).astype(np.float32)
    from mica_b200.pdb import CHANNEL_NAMES
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, 'resampled_normalized_map.mrc')
        rh._write_mrc(p, vol)
        gp = os.path.join(td, 'grids', 'id')
        n, offset, cubes, orig_shape = rh.grids_from_mrc(
            p, os.path.join(gp, 'normalized_map_grids'), prefix='normalized_map_grid')
        for c, name in enumerate(CHANNEL_NAMES):
            pc = os.path.join(td, f'{name}_encoding.mrc')
            rh._write_mrc(pc, enc[c])
            rh.grids_from_mrc(pc, os.path.join(gp, 'AF3_encoding_grids', f'{name}_grids'),
                              prefix=f'{name}_grid')
        keys = sorted(cubes)
        bb, ca, aa = synthetic.synthetic_logits(len(keys), 64, seed=99)
        table = {cubes[k][0].tobytes(): (bb[n_], ca[n_], aa[n_]) for n_, k in enumerate(keys)}
        ok, vols = rh.predict_and_stitch(gp, os.path.join(td, 'out'), table, batch_threshold=1)
        assert ok and len(vols) == 4
    meta = np.array([(k + cubes[k][1:]) for k in keys], dtype=np.int64)
    o = orc.postprocess_and_stitch(bb, ca, aa, meta, orig_shape)
    for name in vols:
        assert np.array_equal(o[name], vols[name]), name
    # float volumes as byte planes and the argmax as uint8 (lossless; tests/_golden.py reads them back):
    # plain float32 deflates to just over 1 MB
    packed = {k + '_planes': byte_planes(v) for k, v in vols.items() if k != 'amino_acid_prediction'}
    _save('stitch.npz', meta=meta, orig_shape=np.array(orig_shape), logits_seed=np.int64(99),
          amino_acid_prediction=vols['amino_acid_prediction'].astype(np.uint8), **packed)


CANDIDATE_CASES = [dict(shape=(56, 44, 40), n_residues=(60, 25), seed=1, wall_margin=3.0),
                   dict(shape=(40, 64, 48), n_residues=(30, 30, 20), seed=2, wall_margin=3.0),
                   dict(shape=(70, 30, 34), n_residues=(90,), seed=3, wall_margin=0.0)]


def golden_candidates():
    """N1: the unmodified Solver.clustering (utils/modeler.py:762-899) on synthetic stitched volumes; the
    inputs are regenerated from the recipe, the reference's outputs are stored."""
    out = {}
    for n, case in enumerate(CANDIDATE_CASES):
        p = synthetic.synthetic_predictions(case['shape'], case['n_residues'], seed=case['seed'],
                                            wall_margin=case['wall_margin'])
        ca, bb = p['carbon_alpha_probability'], p['backbone_probability']
        aa, ap = p['amino_acid_probability'], p['amino_acid_prediction']
        r = rh.solver_clustering(ca, bb, aa, ap)
        o = cand_orc.ca_candidates(ca, bb, aa, ap)
        vp = o['points'][o['valid']]
        sc = ca[vp[:, 0], vp[:, 1], vp[:, 2]]
        assert len(np.unique(sc)) == len(sc), 'ties among the scores: the reference order is undefined'
        for k in ('CA_cands', 'CA_cands_AAProb', 'CA_cands_AA', 'CAProb_clusted'):
            assert np.array_equal(r[k], o[k]), (n, k)
        d, nm, best = cand_orc.neighbor_scores(o['CA_cands'], bb)
        assert np.array_equal(d, r['cand_self_dis']) and np.array_equal(nm, r['neigh_mat']) and best == r['best_neigh']
        for key, lst in cand_orc.neighbor_scores.lists.items():
            assert all(np.array_equal(x, y) for x, y in zip(lst, r[key])) and len(lst) == len(r[key]), key
        for row in nm:                                   # the two best scores of a row must not tie (unstable argsort)
            top = np.sort(row[row > 0])[-3:]
            assert len(np.unique(top)) == len(top)
        print(f'    case {n}: {len(o["points"])} points, {int(o["labels"].max()) + 1} clusters, '
              f'{len(o["picks"])} picks, {int((~o["picks_kept"]).sum())} on the border')
        out.update({f'c{n}_CA_cands': r['CA_cands'], f'c{n}_CA_cands_AAProb': r['CA_cands_AAProb'],
                    f'c{n}_CA_cands_AA': r['CA_cands_AA'],
                    f'c{n}_clusted_lin': np.flatnonzero(r['CAProb_clusted']).astype(np.int64),
                    f'c{n}_labels': o['labels'].astype(np.int32), f'c{n}_picks': o['picks'],
                    f'c{n}_ca_crc': np.float64(ca.astype(np.float64).sum()),
                    f'c{n}_neigh_mat': r['neigh_mat'].astype(np.float64),
                    f'c{n}_cand_self_dis': r['cand_self_dis'].astype(np.float64),
                    f'c{n}_best_neigh': np.array([b + [-1] * (2 - len(b)) for b in r['best_neigh']], dtype=np.int32),
                    **{f'c{n}_{key}_flat': np.concatenate(r[key]).astype(np.int32) for key in cand_orc.neighbor_scores.lists},
                    **{f'c{n}_{key}_len': np.array([len(x) for x in r[key]], dtype=np.int32)
                       for key in cand_orc.neighbor_scores.lists}})
    _save('candidates.npz', n_cases=np.int64(len(CANDIDATE_CASES)), **out)


def _mask_case():
    shape = (40, 36, 32)                                             # (nz, ny, nx): z beyond nx-1 is mis-clamped (D7)
    origin = (np.float32(-2.5), np.float32(3.25), np.float32(1.0))
    st = synthetic.synthetic_structure(160, (32, 36, 40), seed=5, origin_xyz=origin, hetero_every=7, unknown_every=11)
    return shape, origin, st


def golden_label_masks():
    """N3: the three unmodified mask generators on a non-cubic map."""
    shape, origin, st = _mask_case()
    with tempfile.TemporaryDirectory() as td:
        mp, pp = os.path.join(td, 'norm.mrc'), os.path.join(td, 's.pdb')
        rh._write_mrc(mp, np.zeros(shape, np.float32), (1, 1, 1), origin)
        synthetic.write_pdb(pp, st)
        bb, ca, aa = rh.label_masks(mp, pp)
    pos = mask_orc.atom_positions(st['coords'], origin, shape)
    names, resn = np.array(st['atom_names']), np.array(st['res_names'])
    assert np.array_equal(bb, mask_orc.atom_class_mask(pos, np.isin(names, ['N', 'CA', 'C', 'O']), shape))
    assert np.array_equal(ca, mask_orc.atom_class_mask(pos, names == 'CA', shape))
    sel = [i for i in range(len(names)) if names[i] == 'CA' and resn[i] in mask_orc.AA_LABELS]
    labs = [mask_orc.AA_LABELS[resn[i]] for i in sel]
    assert np.array_equal(aa, mask_orc.amino_acid_mask(pos[sel], labs, shape))
    assert np.array_equal(aa, mask_orc.amino_acid_mask_closed_form(pos[sel], labs, shape))
    _save('label_masks.npz', backbone=bb.astype(np.int8), carbon_alpha=ca.astype(np.int8), amino_acid=aa.astype(np.int8))


def golden_docking_masks():
    """N4: initial_map_processing + subsequent_map_processing, isotropic and anisotropic voxels."""
    shape, origin, _ = _mask_case()
    src = synthetic.synthetic_map(shape, seed=3)
    out = {}
    with tempfile.TemporaryDirectory() as td:
        pp = os.path.join(td, 's.pdb')
        for n, (vox, radius) in enumerate([((1.0, 1.0, 1.0), 2.0), ((1.06, 0.93, 1.2), 3.3), ((0.83, 0.83, 0.83), 2.0),
                                           ((0.5, 0.5, 0.5), 2.0)]):
            box = (31 * vox[0], 35 * vox[1], 31 * vox[2])
            st = synthetic.synthetic_structure(120, box, seed=5, origin_xyz=origin, hetero_every=7)
            synthetic.write_pdb(pp, st)
            thr, masked, vs = rh.docking_masks(src, vox, origin, pp, td, 0.1, radius=radius)
            o_thr = mask_orc.contour_threshold(src, 0.1)
            sel = mask_orc.select_central_atoms(st['coords'])
            assert np.array_equal(thr, o_thr)
            assert np.array_equal(masked, mask_orc.mask_around_atoms(o_thr, sel, vs, origin, radius))
            assert np.array_equal(masked, mask_orc.mask_around_atoms_restated(o_thr, sel, vs, origin, radius))
            out.update({f'd{n}_voxel': np.array(vs, np.float32), f'd{n}_box': np.array(box), f'd{n}_radius': np.float64(radius),
                        f'd{n}_zeroed': np.flatnonzero(masked != thr).astype(np.int64)})
    _save('docking_masks.npz', n_cases=np.int64(4), thr_nonzero=np.flatnonzero(o_thr).astype(np.int64), **out)


def main():
    assert rh.available(), 'needs /root/reference'
    os.makedirs(GOLDEN, exist_ok=True)
    only = sys.argv[1:]
    for fn in (golden_preprocess, golden_af3_cubic, golden_cubes, golden_training_twins, golden_stitch,
               golden_candidates, golden_label_masks, golden_docking_masks):
        if only and fn.__name__ not in only:
            continue
        print(fn.__name__)
        fn()


if __name__ == '__main__':
    main()
