"""pfb_model_from_files (C-ABI, pyflyt_b200/csrc/pfb_model_files.cu): URDF + parameter YAML -> PfbModel without Python.
Checked field by field against the Python table builder (pyflyt_b200/models/{urdf,tables}.py, itself checked against
SURVEY.md A.2 in tests/test_models.py) on synthetic vehicles written here — rotated joint / inertial / collision frames,
comments, a stray tail after </robot>, scalar and list PID gains — and on the original PyFlyt's own five vehicle
descriptions (URDF + YAML, stored unmodified under tests/golden/vehicles)."""
import os

import pytest

from pyflyt_b200._lib import PfbError
from pyflyt_b200.models.tables import build_model, model_from_files, model_to_dict

REF_MODELS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vehicles")


def _link(name, mass, ixyz=(0, 0, 0), irpy=(0, 0, 0), inertia=(0, 0, 0, 0, 0, 0), collision=""):
    ixx, iyy, izz, ixy, ixz, iyz = inertia
    return f"""
  <link name="{name}">
    <inertial>
      <origin xyz="{ixyz[0]} {ixyz[1]} {ixyz[2]}" rpy="{irpy[0]} {irpy[1]} {irpy[2]}"/>
      <mass value="{mass}"/>
      <inertia ixx="{ixx}" ixy="{ixy}" ixz="{ixz}" iyy="{iyy}" iyz="{iyz}" izz="{izz}"/>
    </inertial>{collision}
  </link>"""


def _joint(name, parent, child, xyz, rpy=(0, 0, 0)):
    return f"""
  <joint name="{name}" type="fixed">
    <parent link="{parent}"/> <child link="{child}"/>
    <origin rpy="{rpy[0]} {rpy[1]} {rpy[2]}" xyz="{xyz[0]} {xyz[1]} {xyz[2]}"/>
  </joint>"""


BOX = """
    <collision>
      <origin xyz="0.01 -0.02 0.03" rpy="0.1 0.2 0.3"/>
      <geometry><box size="0.2 0.1 0.05"/></geometry>
    </collision>"""
CYL = """
    <collision>
      <origin xyz="0 0 -0.4" rpy="0 0 0.5"/>
      <geometry>
        <cylinder radius="0.12" length="0.9"/>
      </geometry>
    </collision>"""
SPH = """
    <collision><geometry><sphere radius="0.07"/></geometry></collision>
    <collision><geometry><mesh filename="ignored.obj"/></geometry></collision>"""


def _write(tmp_path, name, links, joints, yaml_text):
    d = tmp_path / name
    d.mkdir()
    urdf = f"""<?xml version="1.0" ?>
<!-- synthetic vehicle for tests/test_model_files.py -->
<robot name="{name}">{''.join(links)}{''.join(joints)}
  <!-- a comment with a <tag> inside -->
</robot>
</robot>
"""
    (d / f"{name}.urdf").write_text(urdf)
    (d / f"{name}.yaml").write_text(yaml_text)
    return str(d / f"{name}.urdf"), str(d / f"{name}.yaml")


QUAD_YAML = """# a comment line
motor_params:
  total_thrust: 3.5   # trailing comment
  thrust_coef: 2.5e-10
  torque_coef: 6.0e-12
  noise_ratio: 0.03
  tau: 0.02

drag_params:
  drag_coef_xyz: 2.0
  drag_area_xyz: 5.0e-4
  drag_coef_pqr: 2.0e-4

control_params:
  ang_vel:
    description: "input: angular velocity command | output: torque # not a comment"
    kp: [3.0e-2, 3.5e-2, 7.0e-2]
    ki: [1.0e-7, 2.0e-7,
         3.0e-4]
    kd: [1.0e-4, 1.0e-4, 0.0]
    lim: [1.0, 1.0, 1.0]
  ang_pos:
    kp: [2.0, 2.1, 2.2]
    ki: [0.0, 0.0, 0.0]
    kd: [0.0, 0.0, 0.0]
    lim: [3.0, 3.0, 3.0]
  lin_vel:
    kp: [0.8, 0.7]
    ki: [0.3, 0.2]
    kd: [0.5, 0.4]
    lim: [0.4, 0.4]
  lin_pos:
    kp: [1.0, 1.1]
    ki: [0.0, 0.0]
    kd: [0.0, 0.0]
    lim: [2.0, 2.0]
  z_pos:
    kp: 1.5
    ki: 0.0
    kd: 0.0
    lim: 1.0
  z_vel:
    kp: 2.5
    ki: 0.5
    kd: 0.05
    lim: 1.0
"""

SURFACE = """
  Cl_alpha_2D: 6.1
  chord: {chord} # meters
  span: {span}
  flap_to_chord: 0.3
  eta: 0.65
  alpha_0_base: -2
  alpha_stall_P_base: +14
  alpha_stall_N_base: -9
  Cd_0: 0.01
  deflection_limit: {defl}
  tau: 0.05
"""
WING_YAML = ("motor_params:\n  total_thrust: 18\n  thrust_coef: 3.16e-10\n  torque_coef: 7.94e-12\n  noise_ratio: 0.02\n  tau: 0.01\n"
             + "main_wing_params:" + SURFACE.format(chord=0.3, span=1.6, defl=0)
             + "left_wing_flapped_params:" + SURFACE.format(chord=0.3, span=0.3, defl=30)
             + "right_wing_flapped_params:" + SURFACE.format(chord=0.3, span=0.3, defl=30)
             + "horizontal_tail_params:" + SURFACE.format(chord=0.2, span=0.625, defl=20)
             + "vertical_tail_params:" + SURFACE.format(chord=0.25, span=0.3, defl=15))
ROCKET_YAML = """booster_params:
  total_fuel: 300.5
  max_fuel_rate: 1.2
  inertia_ixx: 1500
  inertia_iyy: 1500
  inertia_izz: 6.5
  min_thrust: 2000.0
  max_thrust: 7000.0
  reignitable: true
  gimbal_range_degrees: 4
  booster_tau: 0.01
  gimbal_tau: 0.02
  noise_ratio: 0.01
finlet_params:""" + SURFACE.format(chord=0.5, span=0.5, defl=45) + """body_params:
  drag_coef_x: 1.1
  drag_coef_y: 1.2
  drag_coef_z: 2.0
  area_x: 1.7
  area_y: 1.6
  area_z: 0.11
"""


def _quad(tmp_path):
    links = [_link("base", 0.8, (0.01, -0.02, 0.005), (0.05, -0.04, 0.3), (0.01, 0.012, 0.016, 1e-4, -2e-4, 3e-4), BOX + SPH)]
    joints = []
    for k, (x, y) in enumerate([(0.16, -0.16), (-0.16, 0.16), (0.16, 0.16), (-0.16, -0.16)]):
        links.append(_link(f"motor{k}", 0.02, (0.0, 0.0, 0.01), (0, 0, 0.1 * k), (1e-5, 1e-5, 2e-5, 0, 0, 0), CYL if k == 0 else ""))
        joints.append(_joint(f"j{k}", "base", f"motor{k}", (x, y, 0.02), (0.0, 0.02 * k, 0.1)))
    links.append(_link("body", 0.0))
    joints.append(_joint("jb", "motor0", "body", (-0.16, 0.16, -0.02), (0.3, 0.0, 0.0)))  # a child of a child
    return _write(tmp_path, "testquad", links, joints, QUAD_YAML)


def _wing(tmp_path):
    names = ["motor", "htail", "vtail", "ail_l", "ail_r", "main"]
    at = [(0, 0, 0), (-1.1, 0, 0), (-1.1, 0, 0.15), (-0.5, 0.95, 0), (-0.5, -0.95, 0), (-0.5, 0, 0.02)]
    mass = [0.0, 0.1, 0.05, 0.2, 0.2, 1.5]
    links = [_link("base", 0.3, collision=BOX)]
    joints = []
    for n, a, m in zip(names, at, mass):
        links.append(_link(n, m, collision=BOX if n in ("main", "htail") else ""))
        joints.append(_joint("j_" + n, "base", n, a))
    return _write(tmp_path, "testwing", links, joints, WING_YAML)


def _rocket(tmp_path):
    links = [_link("base", 91.0, inertia=(500.0, 500.0, 3.0, 0, 0, 0), collision=CYL),
             _link("tank", 0.0), _link("booster", 47.0, inertia=(192.43, 192.43, 0.81, 0, 0, 0), collision=CYL)]
    joints = [_joint("jt", "base", "tank", (0, 0, 0)), _joint("jbo", "base", "booster", (0, 0, -2.0))]
    for k, (x, y) in enumerate([(0.35, 0), (-0.35, 0), (0, 0.35), (0, -0.35)]):
        links.append(_link(f"fin{k}", 0.05, collision=BOX))
        joints.append(_joint(f"jf{k}", "base", f"fin{k}", (x, y, 2.051), (0, 0, 1.5707963 * (k // 2))))
    return _write(tmp_path, "testrocket", links, joints, ROCKET_YAML)


def _assert_same(a, b, path=""):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), path
        for k in a:
            _assert_same(a[k], b[k], f"{path}.{k}")
    elif isinstance(a, list):
        assert len(a) == len(b), path
        for i, (x, y) in enumerate(zip(a, b)):
            _assert_same(x, y, f"{path}[{i}]")
    elif isinstance(a, float):
        assert abs(a - b) <= 1e-12 * max(1.0, abs(a)), (path, a, b)
    else:
        assert a == b, (path, a, b)


@pytest.mark.parametrize("kind,maker", [("quadx", _quad), ("fixedwing", _wing), ("rocket", _rocket)])
def test_c_loader_equals_python_table_builder(tmp_path, kind, maker):
    urdf, yml = maker(tmp_path)
    name = os.path.basename(os.path.dirname(urdf))
    py = build_model(kind, name, model_dir=str(tmp_path))
    c = model_from_files(kind, urdf, yml)
    _assert_same(model_to_dict(py), model_to_dict(c))
    assert c.n_shapes >= 2 and c.mass > 0
    # other rates / constructor options
    py = build_model(kind, name, model_dir=str(tmp_path), physics_hz=480, control_hz=60, starting_velocity=[15.0, 1.0, 0.0], starting_fuel_ratio=0.5)
    c = model_from_files(kind, urdf, yml, physics_hz=480, control_hz=60, starting_velocity=[15.0, 1.0, 0.0], starting_fuel_ratio=0.5)
    _assert_same(model_to_dict(py), model_to_dict(c))


@pytest.mark.parametrize("kind,name", [("quadx", "cf2x"), ("quadx", "primitive_drone"), ("fixedwing", "fixedwing"), ("fixedwing", "acrowing"),
                                       ("rocket", "rocket")])
def test_c_loader_on_the_reference_vehicles(kind, name):
    urdf, yml = os.path.join(REF_MODELS, name, f"{name}.urdf"), os.path.join(REF_MODELS, name, f"{name}.yaml")
    c = model_to_dict(model_from_files(kind, urdf, yml))
    _assert_same(model_to_dict(build_model(kind, name, model_dir=REF_MODELS)), c)  # the Python parser on the same files
    _assert_same(model_to_dict(build_model(kind, name)), c)                        # the package's own committed table


def test_c_loader_errors(tmp_path):
    urdf, yml = _quad(tmp_path)
    with pytest.raises(PfbError, match="cannot read URDF"):
        model_from_files("quadx", str(tmp_path / "nope.urdf"), yml)
    with pytest.raises(PfbError, match="cannot read parameter file"):
        model_from_files("quadx", urdf, str(tmp_path / "nope.yaml"))
    with pytest.raises(PfbError, match="must be multiple of"):  # base_drone.py:94-97
        model_from_files("quadx", urdf, yml, physics_hz=240, control_hz=100)
    bad = tmp_path / "bad.urdf"
    bad.write_text(open(urdf).read().replace('type="fixed"', 'type="revolute"', 1))
    with pytest.raises(PfbError, match="every joint must be 'fixed'"):
        model_from_files("quadx", str(bad), yml)
    bad.write_text("<robot name='x'><link name='a'></robot>")
    with pytest.raises(PfbError, match="XML error"):
        model_from_files("quadx", str(bad), yml)
    short = tmp_path / "short.yaml"
    short.write_text("motor_params:\n  total_thrust: 2.0\n")
    with pytest.raises(PfbError, match="missing parameter `motor_params.thrust_coef`"):
        model_from_files("quadx", urdf, str(short))
    stub_urdf, stub_yaml = _write(tmp_path, "stub", [_link("base", 1.0)], [], ROCKET_YAML)
    with pytest.raises(PfbError, match="vehicle has no link 0"):  # a rocket table needs the tank / booster / finlet links
        model_from_files("rocket", stub_urdf, stub_yaml)
