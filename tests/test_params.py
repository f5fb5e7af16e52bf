"""Parameters under the reference's own names: qlb_params_set_key / qlb_params_from_yaml (host code, runs without
a GPU) and the adapter classes' loadParameters() (GPU)."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from quadruped_locomotion_b200 import build, capi

YAML = """
# a file in the layout of balance_controller/config/controller_gains.yaml
balance_controller:
  virtual_model_controller:
    heading: {}
    lateral:
      kp: 4321.5   # trailing comment
      kd: 4000
      kff: 10
    vertical:
      kp: 10000
      kd: 5000
      kff: 100
    roll:
      kp: 10000
      kd: 1000
      kff: 0.2
    pitch:
      kp: 10000
      kd: 1000
      kff: 0.2
    yaw:
      kp: 4000
      kd: 1000
      kff: 1e3
  contact_force_distribution:
    weights:
      force:
        heading: 2
        lateral: 5
        vertical: 1
      torque:
        roll: 10
        pitch: 10
        yaw: 7.5
      regularizer:
        value: 0.0002
    constraints:
      friction_coefficient: 0.45
      minimal_normal_force: 12
single_leg_controller:
  x_direction:
    kp: 300
"""


def test_keys_are_the_references_parameter_paths(qlb_built):
    lib = capi.load()
    n = lib.qlb_params_num_keys()
    keys = [lib.qlb_params_key(i).decode() for i in range(n)]
    assert n == 27 and len(set(keys)) == n
    assert "/balance_controller/contact_force_distribution/weights/regularizer/value" in keys
    assert "/balance_controller/virtual_model_controller/yaw/kff" in keys
    p = capi.default_params()
    for i, k in enumerate(keys):
        v = C.c_double()
        assert lib.qlb_params_get_key(C.byref(p), k.encode(), C.byref(v)) == i
        assert lib.qlb_params_set_key(C.byref(p), k.encode(), v.value + 1.0) == i
        v2 = C.c_double()
        lib.qlb_params_get_key(C.byref(p), k.encode(), C.byref(v2))
        assert v2.value == v.value + 1.0
    assert lib.qlb_params_set_key(C.byref(p), b"/balance_controller/nope", 1.0) < 0
    assert lib.qlb_params_key(n) is None


def test_yaml_fills_the_parameter_block(qlb_built):
    p, missing = capi.params_from_yaml(YAML)
    # heading gains are not in the file: the reference's loadParameters() would refuse to start
    assert missing == "/balance_controller/virtual_model_controller/heading/kp"
    assert list(p.wrench_weights) == [2.0, 5.0, 1.0, 10.0, 10.0, 7.5]
    assert p.ground_force_weight == 0.0002 and p.friction_default == 0.45 and p.min_normal_force == 12.0
    assert p.kp_translation[1] == 4321.5 and p.kff_rotation[2] == 1000.0
    assert p.kp_translation[0] == 5000.0      # untouched default
    full = YAML.replace("heading: {}", "heading:\n      kp: 1\n      kd: 2\n      kff: 3")
    p, missing = capi.params_from_yaml(full)
    assert missing is None and [p.kp_translation[0], p.kd_translation[0], p.kff_translation[0]] == [1.0, 2.0, 3.0]


def _yaml(tree: dict, indent: str = "") -> str:
    return "".join(f"{indent}{k}:\n" + _yaml(v, indent + "  ") if isinstance(v, dict) else f"{indent}{k}: {v!r}\n"
                   for k, v in tree.items())


def test_defaults_are_the_references_file(qlb_built):
    """The values of the reference's controller_gains.yaml (tests/golden/controller_gains.json, written out again in
    the file's layout) reproduce qlb_default_params exactly."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "controller_gains.json")) as f:
        text = _yaml(json.load(f)["parameters"])
    p0 = capi.default_params()
    zero = capi.default_params()
    lib = capi.load()
    for i in range(lib.qlb_params_num_keys()):
        lib.qlb_params_set_key(C.byref(zero), lib.qlb_params_key(i), -1.0)
    p, missing = capi.params_from_yaml(text, base=zero)
    assert missing is None
    assert bytes(p) == bytes(p0)


@pytest.mark.gpu
def test_adapter_load_parameters(qlb_built):
    demo = build.build_host_demo(which="params_demo")
    r = subprocess.run([demo], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    rows = [ln.split() for ln in r.stdout.strip().splitlines()]
    assert rows[0] == ["loaded", "1", "1"]
    fz = np.array([float(v) for v in rows[1][1:]])
    assert (fz >= 25.0 - 1e-9).all() and abs(fz.sum() - 499.8) < 5.0      # F_min = 25 from the file; the hundredfold
    # regulariser of the file pulls the total a little below the commanded 499.8 N
    assert [float(v) for v in rows[2][1:]] == [0.01, 25.0, 0.3, 12000.0]
    assert rows[3][:2] == ["missing", "1"] and rows[3][2].endswith("/weights/torque/pitch")
    assert rows[4] == ["refused", "1"]
