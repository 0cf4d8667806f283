"""bfloat16 inference, host side: ``precision=`` / ``MICA_PRECISION`` parsing and refusals, the dtype checks that run
before any allocation or launch, the C ABI's refusal of other dtype codes, and the logits hand-off ``_f32c``."""
import ctypes as C

import pytest
import torch

from mica_b200 import _lib, ops
from mica_b200.pipeline import MapPipeline, _f32c
from mica_b200.predict import CryoEMPredictor, parse_precision


@pytest.mark.parametrize('spec,want', [(None, torch.float32), ('', torch.float32), ('  ', torch.float32),
                                       ('fp32', torch.float32), ('bf16', torch.bfloat16), (' BF16 ', torch.bfloat16),
                                       ('FP32', torch.float32)])
def test_parse_precision(spec, want):
    assert parse_precision(spec) is want


@pytest.mark.parametrize('bad', ['fp16', 'bfloat16x', 'half', 16, 2.0, True, torch.bfloat16, ['bf16']])
def test_parse_precision_refusals(bad):
    with pytest.raises(ValueError):
        parse_precision(bad)


def test_predictor_refuses_a_bad_precision_before_any_launch(tmp_path, monkeypatch):
    monkeypatch.delenv('MICA_PRECISION', raising=False)
    n0 = ops.launch_count()
    for kw, env in (({'precision': 'fp16'}, None), ({}, 'int8'), ({'precision': 3}, 'bf16')):
        if env is None:
            monkeypatch.delenv('MICA_PRECISION', raising=False)
        else:
            monkeypatch.setenv('MICA_PRECISION', env)
        pr = CryoEMPredictor('unused', str(tmp_path / 'grids') + '/', str(tmp_path / 'out'), save_output=False,
                             quiet=True, model=lambda x, af: None, **kw)
        pr.logger.disabled = True
        assert pr.run_prediction() == (False, {})
    assert ops.launch_count() == n0


def test_explicit_precision_wins_over_the_environment(monkeypatch):
    monkeypatch.setenv('MICA_PRECISION', 'bf16')
    pr = CryoEMPredictor('unused', 'g/', 'o', model=lambda x, af: None, precision='fp32')
    assert pr._resolve_precision() is torch.float32
    pr = CryoEMPredictor('unused', 'g/', 'o', model=lambda x, af: None)
    assert pr._resolve_precision() is torch.bfloat16


def test_model_fn_wraps_only_bf16():
    model = lambda x, af: (x, af)                                     # noqa: E731
    pr = CryoEMPredictor('unused', 'g/', 'o', model=model)
    assert pr._model_fn(model) is model
    pr._cube_dtype = torch.bfloat16
    assert pr._model_fn(model) is not model


@pytest.mark.parametrize('dt', [torch.float16, torch.float64, torch.int8, 'bf16', None])
def test_cube_dtype_refused_before_any_allocation(dt):
    with pytest.raises(_lib.MicaError, match='float32 or torch.bfloat16'):
        MapPipeline('cuda', cube_dtype=dt)
    with pytest.raises(_lib.MicaError, match='float32 or torch.bfloat16'):
        ops.Af3CubeFiller('cpu', 4, dtype=dt)


def test_model_dtypes():
    assert ops.model_dtype(torch.bfloat16) is torch.bfloat16 and ops.model_dtype(torch.float32) is torch.float32
    assert ops.MODEL_DTYPES == {torch.float32: _lib.DTYPE_F32, torch.bfloat16: _lib.DTYPE_BF16}
    assert _lib.DTYPE_BF16 not in (0, 1, 2, 3, 4, 6, 12, 101)         # not an MRC2014 mode


def test_f32c_passes_float32_and_bfloat16_through():
    a, b = torch.ones((2, 4, 3)), torch.ones((2, 4, 3), dtype=torch.bfloat16)
    for t in (a, b):
        out = _f32c(t, t, t)
        assert all(o is t for o in out)
    nc = torch.ones((4, 2, 3), dtype=torch.bfloat16).transpose(0, 1)
    out = _f32c(nc, nc, nc)
    assert all(o.dtype == torch.bfloat16 and o.is_contiguous() and torch.equal(o, nc) for o in out)
    h = torch.ones((2, 3), dtype=torch.float16)
    assert all(o.dtype == torch.float32 for o in _f32c(h, h, h))
    mixed = _f32c(b, a, b)                                            # a mix becomes float32, as before
    assert all(o.dtype == torch.float32 for o in mixed)


def _as_calls(dtype):
    """Every *_as entry point with null pointers and ``dtype``: the dtype is checked first, on the host."""
    lib, p, i3 = _lib.lib, None, _lib.int3((0, 1, 2))
    w = (C.c_float * 1)(1.0)
    return {
        'extract': lambda: lib.mica_extract_cubes_as(p, 0, 1, 8, 8, 8, 0, 8, i3, 8, 0, p, 1, p, dtype, 512, p, p, 0, p),
        'af3_fill': lambda: lib.mica_af3_fill_cubes_as(p, 0, 8, 8, 8, i3, 8, 0, p, 0, p, 1, p, dtype, 512, p, 0, 0, p),
        'stitch': lambda: lib.mica_postproc_stitch_as(p, p, p, dtype, p, 1, 8, 8, 8, i3, i3, 8, 0, p, p, p, p, p),
        'stitch_peer': lambda: lib.mica_postproc_stitch_peer_as(p, p, p, dtype, p, 1, 8, 8, 8, 8, 0, p, i3, 1, p),
        'overlap': lambda: lib.mica_overlap_accumulate_fixed_as(p, p, p, dtype, p, 1, 8, 8, 8, 8, 0, w, p, 0, p, p),
        'overlap_peer': lambda: lib.mica_overlap_accumulate_fixed_peer_as(p, p, p, dtype, p, 1, 8, 8, 8, 8, 0, w, p, 0,
                                                                          p, 0, i3, 1, p),
    }


@pytest.mark.parametrize('dtype', [_lib.DTYPE_I8, _lib.DTYPE_I16, _lib.DTYPE_U16, 3, 12, -1, 17])
def test_abi_refuses_other_dtypes_on_the_host(dtype):
    for name, call in _as_calls(dtype).items():
        assert call() == -1, name                                     # MICA_ERR_INVALID
        assert 'dtype' in _lib.last_error(), name


def test_resample_refuses_bf16():
    lib, p = _lib.lib, None
    rc = lib.mica_resample(p, _lib.DTYPE_BF16, 8, 8, 8, 0, 8, p, _lib.DTYPE_BF16, 8, 8, 8, 0, 8, p, 0, 3, p)
    assert rc == -1 and 'dtype' in _lib.last_error()
