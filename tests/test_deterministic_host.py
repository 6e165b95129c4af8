"""Deterministic training mode, host side: how the switch is read and the C-ABI entry points it adds."""
import re

import pytest

from scann_b200 import _abi
from scann_b200.engine import deterministic_mode
from tests.test_abi import header_symbols

DET_SYMBOLS = ["scann_plan_inverse", "scann_row_gather", "scann_la_backward_pipe_det", "scann_dense_chain2_det",
               "scann_dense_chain2_grid", "scann_wgrad_batch_tc_det", "scann_wgrad_batch_reduce",
               "scann_geom_init_backward_det", "scann_embed_backward_det", "scann_embed_backward_det_slots",
               "scann_ga_head_backward_det", "scann_rmse_prepare_det", "scann_adam_step_det", "scann_slot_reduce",
               "scann_dense_chain_det", "scann_dense_chain_grid", "scann_noupdate_geom_backward_det",
               "scann_cgcnn_embed_backward_det", "scann_adam_p2p_step_det"]


@pytest.mark.parametrize("env,want", [
    ({}, False),
    ({"SCANN_DETERMINISTIC": "1"}, True),
    ({"SCANN_DETERMINISTIC": "0"}, False),
    ({"TF_DETERMINISTIC_OPS": "1"}, True),
    ({"TF_DETERMINISTIC_OPS": "true"}, True),
    ({"TF_DETERMINISTIC_OPS": "True"}, True),
    ({"TF_DETERMINISTIC_OPS": "0"}, False),
    ({"TF_DETERMINISTIC_OPS": "false"}, False),
    ({"TF_DETERMINISTIC_OPS": ""}, False),
    ({"TF_CUDNN_DETERMINISTIC": "1"}, False),
])
def test_switch_read_from_the_environment(env, want):
    assert deterministic_mode(None, env) is want


@pytest.mark.parametrize("env", [{}, {"SCANN_DETERMINISTIC": "1"}, {"TF_DETERMINISTIC_OPS": "true"}])
def test_explicit_argument_overrides_the_environment(env):
    assert deterministic_mode(False, env) is False
    assert deterministic_mode(True, env) is True


def test_switch_reads_os_environ_by_default(monkeypatch):
    monkeypatch.delenv("SCANN_DETERMINISTIC", raising=False)
    monkeypatch.delenv("TF_DETERMINISTIC_OPS", raising=False)
    assert deterministic_mode() is False
    monkeypatch.setenv("TF_DETERMINISTIC_OPS", "1")
    assert deterministic_mode() is True


def test_facade_passes_the_switch_through():
    import inspect
    from scann_b200.engine import Engine
    from scann_b200.model import ScannKerasModel, create_model
    for fn in (Engine.__init__, ScannKerasModel.__init__, create_model):
        p = inspect.signature(fn).parameters["deterministic"]
        assert p.default is None


@pytest.mark.parametrize("name", DET_SYMBOLS)
def test_new_entry_points_declared_exported_and_bound(name):
    assert name in header_symbols()
    assert hasattr(_abi.lib, name)
    assert name in _abi.PROTOTYPES


def test_slot_table_entry_matches_the_header():
    import ctypes
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(_abi.__file__)))
    src = open(os.path.join(root, "include", "scann_b200.h")).read()
    body = re.search(r"typedef struct ScannSlotSum \{(.*?)\} ScannSlotSum;", src, re.S).group(1)
    assert "const float* slots" in body and "float* dst" in body and "int nslots, count, ld, pad" in body
    assert ctypes.sizeof(_abi.SlotSum) == 32
