"""CPU-side checks: the C-ABI library builds, loads and exports what include/crop2seg_b200.h declares; the
drop-in modules keep the reference's constructor / state_dict contract; nothing silently falls back to CPU."""
import ctypes
import os
import re
import sys
import types

import numpy as np
import pytest
import torch

import crop2seg_b200 as c2s
from crop2seg_b200 import _lib
from crop2seg_b200.build import LIB_PATH, build_library
from golden_util import fixture_names, load
from c2s_testlib import module_from_fixture

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    build_library()
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    header = open(os.path.join(ROOT, "include", "crop2seg_b200.h")).read()
    declared = set(re.findall(r"\b(c2s_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS)
    raw = ctypes.CDLL(LIB_PATH)
    for sym in declared:
        assert hasattr(raw, sym), sym
    assert lib.c2s_abi_version() == _lib.C2S_ABI_VERSION == 12


def test_header_compiles_as_plain_c(tmp_path):
    src = tmp_path / "abi.c"
    src.write_text('#include "crop2seg_b200.h"\nint main(void){c2s_agg_desc d; c2s_ltae_desc l; (void)d; (void)l; '
                   'return sizeof(c2s_ltae_params) == 24 * sizeof(void*) && sizeof(c2s_ltae_bwd_io) == 10 * sizeof(void*) ? 0 : 1;}\n')
    exe = tmp_path / "abi"
    import subprocess
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    assert subprocess.run([str(exe)]).returncode == 0
    assert ctypes.sizeof(_lib.AggDesc) == 40 and ctypes.sizeof(_lib.LtaeDesc) == 76
    assert ctypes.sizeof(_lib.LtaeParams) == 24 * ctypes.sizeof(ctypes.c_void_p)
    assert ctypes.sizeof(_lib.LtaeBwdIo) == 10 * ctypes.sizeof(ctypes.c_void_p)


def test_bad_arguments_return_status_codes_not_aborts(lib):
    assert lib.c2s_agg_forward(None, None, None, None, None, None, 0, None) == 1
    assert b"desc is NULL" in lib.c2s_last_error()
    d = _lib.AggDesc(B=1, T=2000, C=4, H=8, W=8, n_heads=1, ha=1, wa=1, mode=_lib.AGG_MEAN, dtype=_lib.F32)
    dummy = ctypes.c_void_p(16)
    assert lib.c2s_agg_forward(ctypes.byref(d), dummy, None, None, dummy, None, 0, None) == 2  # UNSUPPORTED: T
    d.T, d.mode = 4, 7
    assert lib.c2s_agg_forward(ctypes.byref(d), dummy, None, None, dummy, None, 0, None) == 1
    assert b"unknown mode" in lib.c2s_last_error()
    assert lib.c2s_ltae_forward(None, None, None, None, None, None, None, None, None, None, 0, None) == 1


def test_workspace_sizes(lib):
    d = _lib.AggDesc(B=2, T=5, C=8, H=8, W=8, n_heads=4, ha=4, wa=4, mode=_lib.AGG_ATT_GROUP, dtype=_lib.F32)
    order = 2 * 4  # B int32: the sample order of the pipelined kernel (optional) sits behind the maps, 16-byte aligned
    assert lib.c2s_agg_workspace_bytes(ctypes.byref(d)) == order  # the shipped models stage no attention map
    d.mode = _lib.AGG_ATT_MEAN
    assert lib.c2s_agg_workspace_bytes(ctypes.byref(d)) == 2 * 5 * 4 * 4 * 4 + order
    d.mode, d.ha, d.wa, d.H, d.W = _lib.AGG_ATT_GROUP, 8, 8, 4, 4  # AvgPool2d branch
    assert lib.c2s_agg_workspace_bytes(ctypes.byref(d)) == 4 * 2 * 5 * 4 * 4 * 4 + order
    l = _lib.LtaeDesc(B=2, T=61, C=128, H=16, W=16, n_head=16, d_k=4, d_model=256, c_out=128, has_inconv=1,
                      pe_mode=_lib.PE_SINUSOID, pe_abs=0, pos_dtype=0, dtype=_lib.BF16, flags=0, gn_eps=1e-5, bn_eps=1e-5)
    n = lib.c2s_ltae_workspace_bytes(ctypes.byref(l))
    assert n >= 2 * 61 * 256 * 4 and n % 256 == 0


REFERENCE_STATE_DICT = {  # SURVEY.md section 8b, probed from the reference
    "inconv.weight": (256, 128, 1), "inconv.bias": (256,), "attention_head.Q": (16, 1, 4),
    "attention_head.fc1_k.weight": (64, 256), "attention_head.fc1_k.bias": (64,),
    "in_norm.weight": (128,), "in_norm.bias": (128,), "out_norm.weight": (128,), "out_norm.bias": (128,),
    "mlp.0.weight": (128, 256), "mlp.0.bias": (128,), "mlp.2.weight": (128,), "mlp.2.bias": (128,),
    "mlp.2.running_mean": (128,), "mlp.2.running_var": (128,), "mlp.2.num_batches_tracked": (),
}


def test_state_dict_contract():
    sd = c2s.LTAE().state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == REFERENCE_STATE_DICT
    assert sd["mlp.2.num_batches_tracked"].dtype == torch.int64
    w = c2s.LTAE4WTAE().state_dict()
    assert set(w) == {k for k in REFERENCE_STATE_DICT if not k.startswith(("mlp", "out_norm"))}
    assert tuple(c2s.LTAE(use_doy=True).state_dict()["positional_encoder.fc.weight"].shape) == (16, 365)
    assert tuple(c2s.LTAE(add_linear=True).state_dict()["positional_encoder.fc.weight"].shape) == (256, 256)
    assert tuple(c2s.LTAE(use_abs_rel_enc=True).state_dict()["positional_encoder_abs.fc.weight"].shape) == (16, 365)
    assert list(c2s.TemporalAggregator("att_group").state_dict()) == []
    # model.apply(weight_init) must still find the torch layer types it re-initialises (weight_init.py:14-48)
    kinds = {type(m) for m in c2s.LTAE().modules()}
    assert {torch.nn.Conv1d, torch.nn.Linear, torch.nn.BatchNorm1d, torch.nn.GroupNorm} <= kinds


@pytest.mark.parametrize("name", fixture_names(["ltae_", "wtae_"]))
def test_reference_state_dicts_load(name):
    cfg, _, params, _ = load(name)
    module_from_fixture(cfg, params, device="cpu")  # strict load_state_dict + identical denom attribute


def test_constructor_assertion_and_signature():
    with pytest.raises(AssertionError):
        c2s.LTAE(mlp=[128, 128], d_model=256)  # tae.py:404
    m = c2s.LTAE(in_channels=64, d_model=None, mlp=[64, 32], n_head=4)
    assert m.inconv is None and m.d_model == 64
    import inspect
    assert list(inspect.signature(c2s.LTAE.forward).parameters)[:5] == ["self", "x", "batch_positions", "pad_mask", "return_comp"]
    assert list(inspect.signature(c2s.TemporalAggregator.forward).parameters) == ["self", "x", "pad_mask", "attn_mask"]


def test_cpu_tensors_fail_loudly():
    agg = c2s.TemporalAggregator("mean")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        agg(torch.zeros(1, 2, 4, 4, 4))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        c2s.LTAE(in_channels=32, n_head=4, mlp=[64, 32], d_model=64).eval()(torch.zeros(1, 2, 32, 2, 2),
                                                                            batch_positions=torch.zeros(1, 2))
    with pytest.raises(NotImplementedError):
        c2s.LTAE(in_channels=32, n_head=4, mlp=[64, 32], d_model=64, num_queries=2)(torch.zeros(1, 2, 32, 2, 2))
    with pytest.raises(RuntimeError, match="Class values"):  # F.one_hot's day-of-year range check
        c2s.LTAE(in_channels=32, n_head=4, mlp=[64, 32], d_model=64, use_doy=True).eval()(
            torch.zeros(1, 2, 32, 2, 2), batch_positions=torch.tensor([[3, 365]]))
    assert c2s.TemporalAggregator("bogus")(torch.zeros(1, 1, 1, 1, 1)) is None  # the reference falls through to None


def test_install_swaps_reference_bindings():
    names = ["src", "src.backbones", "src.backbones.tae", "src.backbones.temporal_aggregator", "src.backbones.utae",
             "src.backbones.wtae", "src.backbones.timeunet"]
    saved = {n: sys.modules.get(n) for n in names}
    try:
        for n in names:
            sys.modules[n] = types.ModuleType(n)
        sentinel = object()
        sys.modules["src.backbones.tae"].LTAE = sentinel
        sys.modules["src.backbones.tae"].LTAE4WTAE = sentinel
        sys.modules["src.backbones.utae"].LTAE = sentinel
        sys.modules["src.backbones.utae"].TemporalAggregator = sentinel
        sys.modules["src.backbones.wtae"].LTAE4WTAE = sentinel
        swapped = c2s.install(import_missing=False)
        assert "src.backbones.utae.LTAE" in swapped and "src.backbones.wtae.LTAE4WTAE" in swapped
        assert sys.modules["src.backbones.utae"].LTAE is c2s.LTAE
        assert sys.modules["src.backbones.utae"].TemporalAggregator is c2s.TemporalAggregator
        c2s.uninstall()
        assert sys.modules["src.backbones.utae"].LTAE is sentinel
    finally:
        c2s.uninstall()
        for n, m in saved.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m


# A stand-in for the reference's src/backbones with the same import-time bindings: the model files take the hot-path
# classes by name from tae.py / temporal_aggregator.py (utae.py:8-9, wtae.py:9-10, timeunet.py:4-5).
STAND_IN_REFERENCE = {
    "src/__init__.py": "",
    "src/backbones/__init__.py": "",
    "src/backbones/tae.py": "class LTAE:\n    pass\n\n\nclass LTAE4WTAE:\n    pass\n",
    "src/backbones/temporal_aggregator.py": "class TemporalAggregator:\n    pass\n",
    "src/backbones/utae.py": ("from src.backbones.tae import LTAE\n"
                              "from src.backbones.temporal_aggregator import TemporalAggregator\n"),
    "src/backbones/wtae.py": ("from src.backbones.tae import LTAE4WTAE\n"
                              "from src.backbones.temporal_aggregator import TemporalAggregator\n"),
    "src/backbones/timeunet.py": ("from src.backbones.tae import LTAE\n"
                                  "from src.backbones.temporal_aggregator import TemporalAggregator\n\n\n"
                                  "class TimeUNet_v1:\n    def forward(self, input, batch_positions=None, return_att=False):\n"
                                  "        return input\n"),
}


def test_install_imports_then_uninstall_restores_the_reference_classes(tmp_path):
    """install() doing the importing itself must still remember the reference classes (the model files import
    src.backbones.tae, so saving while importing would record the fused class as the original)."""
    import subprocess
    for rel, text in STAND_IN_REFERENCE.items():
        (tmp_path / rel).parent.mkdir(parents=True, exist_ok=True)
        (tmp_path / rel).write_text(text)
    code = (
        "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
        "import crop2seg_b200 as c2s\n"
        "swapped = c2s.install(assume_zero_padded=True)\n"
        "import src.backbones.utae as u, src.backbones.tae as t, src.backbones.timeunet as tu\n"
        "assert u.LTAE is c2s.LTAE and t.LTAE is c2s.LTAE and tu.LTAE is c2s.LTAE, swapped\n"
        "assert c2s.LTAE().assume_zero_padded is True\n"
        "wrapped = tu.TimeUNet_v1.forward\n"
        "c2s.uninstall()\n"
        "assert t.LTAE.__module__ == 'src.backbones.tae' and u.LTAE is t.LTAE and tu.LTAE is t.LTAE\n"
        "assert u.TemporalAggregator.__module__ == 'src.backbones.temporal_aggregator'\n"
        "assert tu.TimeUNet_v1.forward is not wrapped and c2s.LTAE().assume_zero_padded is False\n"
        "print('ok')\n") % (str(tmp_path), ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "ok" in res.stdout, res.stderr[-2000:]


def test_shard_bounds_partition():
    for n in (0, 1, 7, 64, 7396):
        for w in (1, 2, 3, 8):
            spans = [c2s.shard_bounds(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        c2s.shard_bounds(4, 2, 2)


def test_copy_valid_frames_skips_padding():
    import torch
    from crop2seg_b200 import copy_valid_frames_, valid_lengths
    src = torch.arange(4 * 5 * 3, dtype=torch.float32).reshape(4, 5, 3)
    dst = torch.full_like(src, -1.0)
    lengths = [5, 2, 0, 5]
    n = copy_valid_frames_(dst, src, lengths)
    assert n == (5 + 2 + 0 + 5) * 3 * 4
    for b, L in enumerate(lengths):
        assert torch.equal(dst[b, :L], src[b, :L]) and bool((dst[b, L:] == -1).all())
    copy_valid_frames_(dst, src, lengths, zero_rest=True)
    assert bool((dst[1, 2:] == 0).all()) and bool((dst[2] == 0).all())
    pad = torch.tensor([[False] * 5, [False, False, True, True, True], [True] * 5, [False] * 5])
    assert valid_lengths(pad) == lengths
    bad = torch.tensor([[False, True, False]])
    import pytest
    with pytest.raises(ValueError):
        valid_lengths(bad)
    with pytest.raises(ValueError):
        copy_valid_frames_(dst, src[:, :4], lengths)
