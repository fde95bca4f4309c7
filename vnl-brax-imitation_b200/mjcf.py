"""MJCF subset parser + model compiler (host side, numpy float64 -> fp32 tables).

The reference builds its physics model with dm_control + the MuJoCo compiler
(`envs/rodent.py:39-63`, `envs/humanoid.py:40-54`, `preprocessing/mjx_preprocess.py:75-86`)
and uploads it with `mjx.put_model`.  Neither package exists in this image, so this
module restates the part of the MuJoCo compiler those call sites rely on:

* `<default>` class inheritance, `childclass`, `<freejoint>`, hinge joints, plane / sphere /
  capsule / ellipsoid / box / cylinder geoms (`fromto`, `euler`, `quat`, `zaxis`, `axisangle`),
  `<general>` / `<motor>` joint actuators, explicit `<pair>` contacts.
* dm_control `rescale.rescale_subtree` semantics (only explicitly-set `pos` / `size` /
  `fromto` of worldbody descendants are scaled) -- `envs/rodent.py:48-52`.
* the torque-actuator edit of `envs/rodent.py:41-45`.
* geom -> body mass / inertia compilation, `qpos0`, `qpos_spring`, `dof_invweight0`,
  `body_invweight0`, `stat.meaninertia`, static collision-pair list with MuJoCo's
  priority / solmix parameter mixing.

The compiled `Model` is a bag of numpy arrays; `model_blob.py` serialises it into the
flat blob `include/vnl_b200.h` describes.  The golden check for this module is the
kinematics / COM data inside `clips/transform_snips_groom.p` (tests/test_mjcf_clip.py).
"""
from __future__ import annotations

import copy
import math
import xml.etree.ElementTree as ET
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np

MJ_MINVAL = 1e-15

GEOM_PLANE, GEOM_SPHERE, GEOM_CAPSULE, GEOM_ELLIPSOID, GEOM_CYLINDER, GEOM_BOX = 0, 2, 3, 4, 5, 6
_GEOM_TYPES = {"plane": GEOM_PLANE, "sphere": GEOM_SPHERE, "capsule": GEOM_CAPSULE,
               "ellipsoid": GEOM_ELLIPSOID, "cylinder": GEOM_CYLINDER, "box": GEOM_BOX}
JNT_FREE, JNT_HINGE = 0, 3
SOLVER_CG, SOLVER_NEWTON = 1, 2
DYN_NONE, DYN_FILTER = 0, 2

_DEFAULT_SOLREF = (0.02, 1.0)
_DEFAULT_SOLIMP = (0.9, 0.95, 0.001, 0.5, 2.0)


# --------------------------------------------------------------------------------------
# small quaternion helpers (float64, [w, x, y, z])
# --------------------------------------------------------------------------------------
def quat_mul(a, b):
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return np.array([aw * bw - ax * bx - ay * by - az * bz,
                     aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx,
                     aw * bz + ax * by - ay * bx + az * bw])


def quat_to_mat(q):
    w, x, y, z = q
    return np.array([[w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z]])


def mat_to_quat(m):
    """Rotation matrix -> unit quaternion (w >= 0)."""
    t = np.trace(m)
    if t > 0:
        s = math.sqrt(t + 1.0) * 2
        q = np.array([0.25 * s, (m[2, 1] - m[1, 2]) / s, (m[0, 2] - m[2, 0]) / s, (m[1, 0] - m[0, 1]) / s])
    elif m[0, 0] > m[1, 1] and m[0, 0] > m[2, 2]:
        s = math.sqrt(1.0 + m[0, 0] - m[1, 1] - m[2, 2]) * 2
        q = np.array([(m[2, 1] - m[1, 2]) / s, 0.25 * s, (m[0, 1] + m[1, 0]) / s, (m[0, 2] + m[2, 0]) / s])
    elif m[1, 1] > m[2, 2]:
        s = math.sqrt(1.0 + m[1, 1] - m[0, 0] - m[2, 2]) * 2
        q = np.array([(m[0, 2] - m[2, 0]) / s, (m[0, 1] + m[1, 0]) / s, 0.25 * s, (m[1, 2] + m[2, 1]) / s])
    else:
        s = math.sqrt(1.0 + m[2, 2] - m[0, 0] - m[1, 1]) * 2
        q = np.array([(m[1, 0] - m[0, 1]) / s, (m[0, 2] + m[2, 0]) / s, (m[1, 2] + m[2, 1]) / s, 0.25 * s])
    q = q / np.linalg.norm(q)
    return q if q[0] >= 0 else -q


def axis_angle_quat(axis, angle):
    axis = np.asarray(axis, dtype=np.float64)
    return np.concatenate([[math.cos(0.5 * angle)], axis * math.sin(0.5 * angle)])


def z_to_quat(vec):
    """Quaternion rotating the z axis onto `vec` (MuJoCo mjuu_z2quat)."""
    vec = np.asarray(vec, dtype=np.float64)
    n = np.linalg.norm(vec)
    if n < MJ_MINVAL:
        return np.array([1.0, 0, 0, 0])
    vec = vec / n
    axis = np.cross([0.0, 0.0, 1.0], vec)
    s = np.linalg.norm(axis)
    if s < 1e-10:
        return np.array([1.0, 0, 0, 0]) if vec[2] > 0 else np.array([0.0, 1.0, 0, 0])
    axis = axis / s
    ang = math.atan2(s, vec[2])
    return axis_angle_quat(axis, ang)


def rotate(v, q):
    return quat_to_mat(q) @ np.asarray(v, dtype=np.float64)


# --------------------------------------------------------------------------------------
# XML helpers
# --------------------------------------------------------------------------------------
def _floats(s: Optional[str]) -> Optional[np.ndarray]:
    if s is None:
        return None
    return np.array([float(t) for t in s.split()], dtype=np.float64)


def _fmt(a: Sequence[float]) -> str:
    return " ".join(repr(float(x)) for x in a)


def load_xml(path: str) -> ET.Element:
    return ET.parse(path).getroot()


def rescale_subtree(root: ET.Element, position_factor: float, size_factor: float) -> None:
    """dm_control `rescale.rescale_subtree(root, pf, sf)` on an ElementTree (in place).

    Semantics restated (dm_control is absent): for every child element, an explicitly
    written `fromto` is rescaled about its midpoint, an explicit `pos` is multiplied by
    `position_factor`, an explicit `size` by `size_factor`; recursion only enters
    `worldbody` and `body` elements, so `<default>` classes are never touched
    (reference call site `envs/rodent.py:48-52`, `mjx_preprocess.py:76-80`).
    """
    for child in list(root):
        if child.get("fromto") is not None:
            ft = _floats(child.get("fromto"))
            new_pos = position_factor * 0.5 * (ft[3:] + ft[:3])
            new_size = size_factor * 0.5 * (ft[3:] - ft[:3])
            child.set("fromto", _fmt(np.concatenate([new_pos - new_size, new_pos + new_size])))
        if child.get("pos") is not None:
            child.set("pos", _fmt(_floats(child.get("pos")) * position_factor))
        if child.get("size") is not None and child.tag in ("geom", "site", "camera", "light", "body", "joint"):
            child.set("size", _fmt(_floats(child.get("size")) * size_factor))
        if child.tag in ("body", "worldbody"):
            rescale_subtree(child, position_factor, size_factor)


def expand_replicate(root: ET.Element, degree: bool = True, eulerseq: str = "xyz") -> None:
    """Expand `<replicate count offset euler sep>` (MuJoCo 3.1.2+, `assets/rodent_pair.xml:163`) in place.

    Copy i (i = 0 .. count-1) of the enclosed subtree is placed in the frame (i * offset, euler applied i times) and
    every `name` inside it gets the suffix `sep + i`.  Elements OUTSIDE the body tree that reference a replicated name
    (actuators, sensors, contact pairs / excludes, tendon-free here) are replicated with the same suffix, which is what
    gives rodent_pair nu = 60.  (The file is render-only in the reference -- `train.py:295-320` -- so there is no golden
    for this interpretation; SURVEY assumption U7.)"""
    import copy
    wb = root.find("worldbody")
    if wb is None:
        return
    suffixed: Dict[str, List[str]] = {}

    def rename(el: ET.Element, suf: str, names: set) -> None:
        for e in el.iter():
            n = e.get("name")
            if n is not None:
                names.add(n)
                e.set("name", n + suf)
        for e in el.iter():  # references inside the copy (camera / light targets, ...)
            for k in ("target", "body", "joint", "site", "geom"):
                v = e.get(k)
                if v is not None and v in names:
                    e.set(k, v + suf)

    def expand(parent: ET.Element) -> None:
        for child in list(parent):
            if child.tag == "replicate":
                count = int(child.get("count", "1"))
                sep = child.get("sep", "")
                offset = _floats(child.get("offset")) if child.get("offset") else np.zeros(3)
                step_q = _orientation({"euler": child.get("euler")}, degree, eulerseq) if child.get("euler") else np.array([1.0, 0, 0, 0])
                idx = list(parent).index(child)
                parent.remove(child)
                q, pos = np.array([1.0, 0, 0, 0]), np.zeros(3)
                for i in range(count):
                    for sub in child:
                        cp = copy.deepcopy(sub)
                        names: set = set()
                        suf = f"{sep}{i}"
                        rename(cp, suf, names)
                        for n in names:
                            suffixed.setdefault(n, []).append(n + suf)
                        if cp.tag in ("body", "geom", "site", "camera", "light", "frame"):
                            lp = _floats(cp.get("pos")) if cp.get("pos") else np.zeros(3)
                            lq = _orientation(cp.attrib, degree, eulerseq)
                            for k in ("euler", "axisangle", "xyaxes", "zaxis"):
                                cp.attrib.pop(k, None)
                            cp.set("pos", _fmt(pos + rotate(lp, q)))
                            cp.set("quat", _fmt(quat_mul(q, lq)))
                        parent.insert(idx, cp)
                        idx += 1
                    pos = pos + rotate(offset, q)
                    q = quat_mul(q, step_q)
            else:
                expand(child)

    expand(wb)
    if not suffixed:
        return
    for section in ("actuator", "sensor", "contact", "tendon", "equality"):
        for sec in root.findall(section):
            for el in list(sec):
                refs = [k for k in ("joint", "site", "body", "body1", "body2", "geom", "geom1", "geom2", "objname", "tendon")
                        if el.get(k) in suffixed]
                if not refs:
                    continue
                ncopy = len(suffixed[el.get(refs[0])])
                pos_in_sec = list(sec).index(el)
                sec.remove(el)
                for i in range(ncopy):
                    cp = copy.deepcopy(el)
                    for k in refs:
                        cp.set(k, suffixed[el.get(k)][i])
                    if cp.get("name") is not None:
                        cp.set("name", suffixed[el.get(refs[0])][i].replace(el.get(refs[0]), cp.get("name"), 1)
                               if False else cp.get("name") + suffixed[el.get(refs[0])][i][len(el.get(refs[0])):])
                    sec.insert(pos_in_sec + i, cp)


def torque_actuators(root: ET.Element) -> None:
    """`envs/rodent.py:41-45`: gainprm <- [forcerange[1]], drop biastype / biasprm."""
    for act in root.iter("general"):
        if act.get("forcerange") is None:
            continue  # the <default><general> templates
        fr = _floats(act.get("forcerange"))
        act.set("gainprm", repr(float(fr[1])))
        act.attrib.pop("biastype", None)
        act.attrib.pop("biasprm", None)


# --------------------------------------------------------------------------------------
# defaults
# --------------------------------------------------------------------------------------
_DEFAULT_TAGS = ("joint", "geom", "site", "general", "motor", "position", "velocity", "pair")


class _Defaults:
    """Nested `<default class=...>` tables: class -> tag -> attribute dict."""

    def __init__(self, root: ET.Element):
        self.classes: Dict[str, Dict[str, Dict[str, str]]] = {"main": {t: {} for t in _DEFAULT_TAGS}}
        for d in root.findall("default"):
            self._walk(d, "main", top=True)

    @staticmethod
    def _tag(tag: str) -> str:
        # actuator shortcuts share one default table with <general>
        return "general" if tag in ("motor", "position", "velocity") else tag

    def _walk(self, node: ET.Element, parent: str, top: bool = False) -> None:
        name = "main" if top else node.get("class")
        if not top:
            self.classes.setdefault(name, copy.deepcopy(self.classes[parent]))
        table = self.classes[name]
        for el in node:
            if el.tag == "default":
                continue
            table.setdefault(self._tag(el.tag), {}).update(el.attrib)
        for el in node.findall("default"):
            self._walk(el, name)

    def resolve(self, el: ET.Element, childclass: Optional[str]) -> Dict[str, str]:
        cls = el.get("class") or childclass or "main"
        if cls not in self.classes:
            raise ValueError(f"unknown default class {cls!r}")
        out = dict(self.classes[cls].get(self._tag(el.tag), {}))
        out.update({k: v for k, v in el.attrib.items() if k != "class"})
        return out


# --------------------------------------------------------------------------------------
# compiled model
# --------------------------------------------------------------------------------------
@dataclass
class Model:
    """Compiled constant tables (float64 / int32 numpy).  Names follow mjModel."""
    name: str = ""
    nq: int = 0
    nv: int = 0
    nu: int = 0
    na: int = 0
    nbody: int = 0
    njnt: int = 0
    ngeom: int = 0
    # options
    timestep: float = 0.002
    gravity: np.ndarray = field(default_factory=lambda: np.array([0.0, 0.0, -9.81]))
    tolerance: float = 1e-8
    ls_tolerance: float = 0.01
    impratio: float = 1.0
    solver: int = SOLVER_NEWTON
    iterations: int = 100
    ls_iterations: int = 50
    eulerdamp: bool = True
    meaninertia: float = 1.0
    # names
    body_names: List[str] = field(default_factory=list)
    jnt_names: List[str] = field(default_factory=list)
    geom_names: List[str] = field(default_factory=list)
    act_names: List[str] = field(default_factory=list)
    arrays: Dict[str, np.ndarray] = field(default_factory=dict)

    def __getattr__(self, k):
        arrays = self.__dict__.get("arrays", {})
        if k in arrays:
            return arrays[k]
        raise AttributeError(k)

    def body_id(self, name: str) -> int:
        return self.body_names.index(name)

    def jnt_id(self, name: str) -> int:
        return self.jnt_names.index(name)


def _orientation(attr: Dict[str, str], degree: bool, eulerseq: str = "xyz") -> np.ndarray:
    if "quat" in attr:
        q = _floats(attr["quat"])
        return q / np.linalg.norm(q)
    if "euler" in attr:
        e = _floats(attr["euler"])
        if degree:
            e = np.deg2rad(e)
        q = np.array([1.0, 0, 0, 0])
        for ax, ang in zip(eulerseq, e):
            axis = {"x": [1.0, 0, 0], "y": [0, 1.0, 0], "z": [0, 0, 1.0]}[ax.lower()]
            r = axis_angle_quat(axis, ang)
            q = quat_mul(q, r) if ax.islower() else quat_mul(r, q)
        return q / np.linalg.norm(q)
    if "axisangle" in attr:
        a = _floats(attr["axisangle"])
        ang = np.deg2rad(a[3]) if degree else a[3]
        return axis_angle_quat(a[:3] / np.linalg.norm(a[:3]), ang)
    if "zaxis" in attr:
        return z_to_quat(_floats(attr["zaxis"]))
    if "xyaxes" in attr:
        a = _floats(attr["xyaxes"])
        x = a[:3] / np.linalg.norm(a[:3])
        y = a[3:] - x * np.dot(x, a[3:])
        y = y / np.linalg.norm(y)
        return mat_to_quat(np.stack([x, y, np.cross(x, y)], axis=1))
    return np.array([1.0, 0, 0, 0])


def _geom_volume_inertia(gtype: int, size: np.ndarray):
    """Volume and unit-density diagonal inertia in the geom frame (MuJoCo mjCGeom)."""
    if gtype == GEOM_SPHERE:
        r = size[0]
        v = 4.0 / 3.0 * math.pi * r ** 3
        i = 2.0 / 5.0 * r * r
        return v, np.array([i, i, i]) * v
    if gtype == GEOM_CAPSULE:
        r, h = size[0], 2.0 * size[1]
        v = math.pi * (r * r * h + 4.0 / 3.0 * r ** 3)
        ms = 4.0 * r / (4.0 * r + 3.0 * h)  # sphere share of unit mass
        mc = 1.0 - ms
        ixx = mc * (3 * r * r + h * h) / 12.0
        izz = mc * r * r / 2.0
        si = 2.0 * ms * r * r / 5.0
        ixx += si + ms * h * (3 * r + 2 * h) / 8.0
        izz += si
        return v, np.array([ixx, ixx, izz]) * v
    if gtype == GEOM_ELLIPSOID:
        a, b, c = size[:3]
        v = 4.0 / 3.0 * math.pi * a * b * c
        return v, np.array([b * b + c * c, a * a + c * c, a * a + b * b]) / 5.0 * v
    if gtype == GEOM_BOX:
        a, b, c = size[:3]
        v = 8.0 * a * b * c
        return v, np.array([b * b + c * c, a * a + c * c, a * a + b * b]) / 3.0 * v
    if gtype == GEOM_CYLINDER:
        r, h = size[0], 2.0 * size[1]
        v = math.pi * r * r * h
        return v, np.array([(3 * r * r + h * h) / 12.0, (3 * r * r + h * h) / 12.0, r * r / 2.0]) * v
    return 0.0, np.zeros(3)


def _solimp(vals: Optional[np.ndarray]) -> np.ndarray:
    out = np.array(_DEFAULT_SOLIMP)
    if vals is not None:
        out[: len(vals)] = vals
    return out


def _solref(vals: Optional[np.ndarray]) -> np.ndarray:
    out = np.array(_DEFAULT_SOLREF)
    if vals is not None:
        out[: len(vals)] = vals
    return out


def set_solver(m: Model, solver: Optional[str] = None, iterations: Optional[int] = None,
               ls_iterations: Optional[int] = None) -> Model:
    """The solver overrides the reference envs apply to a compiled model (`envs/rodent.py:55-63`, `envs/humanoid.py:43-54`);
    None keeps the model's value."""
    if solver is not None:
        m.solver = {"cg": SOLVER_CG, "newton": SOLVER_NEWTON}[solver.lower()]
    if iterations is not None:
        m.iterations = int(iterations)
    if ls_iterations is not None:
        m.ls_iterations = int(ls_iterations)
    return m


def compile_model(root: ET.Element, *, name: str = "", solver: Optional[str] = None,
                  iterations: Optional[int] = None, ls_iterations: Optional[int] = None,
                  eulerdamp: Optional[bool] = None) -> Model:
    """Compile an MJCF ElementTree into constant tables.

    `solver / iterations / ls_iterations / eulerdamp` are the post-compile overrides the
    reference envs apply (`envs/rodent.py:55-63`, `envs/humanoid.py:43-54`).
    """
    comp = {}
    for c in root.findall("compiler"):
        comp.update(c.attrib)
    degree = comp.get("angle", "degree") == "degree"
    eulerseq = comp.get("eulerseq", "xyz")
    autolimits = comp.get("autolimits", "true") == "true"
    expand_replicate(root, degree, eulerseq)
    defaults = _Defaults(root)

    m = Model(name=name or root.get("model", ""))
    opt = root.find("option")
    if opt is not None:
        m.timestep = float(opt.get("timestep", m.timestep))
        if opt.get("gravity"):
            m.gravity = _floats(opt.get("gravity"))
        m.tolerance = float(opt.get("tolerance", m.tolerance))
        m.ls_tolerance = float(opt.get("ls_tolerance", m.ls_tolerance))
        m.impratio = float(opt.get("impratio", m.impratio))
        m.iterations = int(opt.get("iterations", m.iterations))
        m.ls_iterations = int(opt.get("ls_iterations", m.ls_iterations))
        if opt.get("solver"):
            set_solver(m, opt.get("solver"))
        if opt.get("cone", "pyramidal") != "pyramidal":
            raise NotImplementedError("only the pyramidal cone is on the reference path")
        flag = opt.find("flag")
        if flag is not None and flag.get("eulerdamp") == "disable":
            m.eulerdamp = False
    set_solver(m, solver, iterations, ls_iterations)
    if eulerdamp is not None:
        m.eulerdamp = bool(eulerdamp)

    bodies: List[dict] = []
    joints: List[dict] = []
    geoms: List[dict] = []

    def add_body(el: ET.Element, parent: int, childclass: Optional[str]) -> None:
        bid = len(bodies)
        is_world = el.tag == "worldbody"
        cc = el.get("childclass") or childclass
        b = dict(name="world" if is_world else el.get("name", f"body{bid}"), parent=parent,
                 pos=np.zeros(3) if is_world else (_floats(el.get("pos")) if el.get("pos") else np.zeros(3)),
                 quat=np.array([1.0, 0, 0, 0]) if is_world else _orientation(el.attrib, degree, eulerseq),
                 joints=[], geoms=[], inertial=None)
        bodies.append(b)
        if el.find("inertial") is not None:
            it = el.find("inertial")
            b["inertial"] = dict(pos=_floats(it.get("pos")), quat=_orientation(it.attrib, degree, eulerseq),
                                 mass=float(it.get("mass")), diag=_floats(it.get("diaginertia")))
        for ch in el:
            if ch.tag in ("joint", "freejoint"):
                if ch.tag == "freejoint":
                    attr = dict(ch.attrib)
                    attr["type"] = "free"
                else:
                    attr = defaults.resolve(ch, cc)
                jt = attr.get("type", "hinge")
                if jt not in ("hinge", "free"):
                    raise NotImplementedError(f"joint type {jt}")
                rng = _floats(attr.get("range")) if attr.get("range") else np.zeros(2)
                lim = attr.get("limited", "auto")
                limited = (lim == "true") or (lim == "auto" and autolimits and attr.get("range") is not None)
                to_rad = (math.pi / 180.0) if (degree and jt == "hinge") else 1.0
                axis = _floats(attr.get("axis")) if attr.get("axis") else np.array([0.0, 0, 1.0])
                j = dict(name=attr.get("name", f"jnt{len(joints)}"), type=JNT_FREE if jt == "free" else JNT_HINGE,
                         body=bid, pos=_floats(attr.get("pos")) if attr.get("pos") else np.zeros(3),
                         axis=axis / np.linalg.norm(axis), range=rng * to_rad,
                         limited=bool(limited) and jt != "free",
                         stiffness=float(attr.get("stiffness", 0.0)), damping=float(attr.get("damping", 0.0)),
                         armature=float(attr.get("armature", 0.0)), margin=float(attr.get("margin", 0.0)),
                         ref=float(attr.get("ref", 0.0)) * to_rad, springref=float(attr.get("springref", 0.0)) * to_rad,
                         solref=_solref(_floats(attr.get("solreflimit"))), solimp=_solimp(_floats(attr.get("solimplimit"))))
                if jt == "free":
                    j.update(stiffness=0.0, limited=False)
                b["joints"].append(len(joints))
                joints.append(j)
            elif ch.tag == "geom":
                attr = defaults.resolve(ch, cc)
                gt = _GEOM_TYPES[attr.get("type", "sphere")]
                size = np.zeros(3)
                if attr.get("size"):
                    s = _floats(attr["size"])
                    size[: len(s)] = s[:3]
                pos = _floats(attr.get("pos")) if attr.get("pos") else np.zeros(3)
                quat = _orientation(attr, degree, eulerseq)
                if attr.get("fromto"):
                    ft = _floats(attr["fromto"])
                    vec = ft[:3] - ft[3:]
                    size[1] = 0.5 * np.linalg.norm(vec)
                    quat = z_to_quat(vec)
                    pos = 0.5 * (ft[:3] + ft[3:])
                fr = np.array([1.0, 0.005, 0.0001])
                if attr.get("friction"):
                    f = _floats(attr["friction"])
                    fr[: len(f)] = f
                g = dict(name=attr.get("name", f"geom{len(geoms)}"), type=gt, body=bid, pos=pos, quat=quat, size=size,
                         contype=int(attr.get("contype", 1)), conaffinity=int(attr.get("conaffinity", 1)),
                         condim=int(attr.get("condim", 3)), priority=int(attr.get("priority", 0)), friction=fr,
                         solref=_solref(_floats(attr.get("solref"))), solimp=_solimp(_floats(attr.get("solimp"))),
                         solmix=float(attr.get("solmix", 1.0)), margin=float(attr.get("margin", 0.0)),
                         gap=float(attr.get("gap", 0.0)), density=float(attr.get("density", 1000.0)),
                         mass=float(attr["mass"]) if attr.get("mass") is not None else None)
                b["geoms"].append(len(geoms))
                geoms.append(g)
            elif ch.tag == "body":
                pass
        for ch in el.findall("body"):
            add_body(ch, bid, cc)

    # MuJoCo numbers bodies depth-first but children AFTER all of a body's own elements;
    # joints/geoms are numbered in body order.  add_body appends a body's own joints/geoms
    # before recursing, which yields exactly that order.
    wb = root.find("worldbody")
    add_body(wb, 0, None)
    # re-number joints and geoms in body order (they were appended depth-first already,
    # but a body's joints may appear in the XML after its child bodies: collect per body).
    jorder = [j for b in bodies for j in b["joints"]]
    gorder = [g for b in bodies for g in b["geoms"]]
    jmap = {old: new for new, old in enumerate(jorder)}
    gmap = {old: new for new, old in enumerate(gorder)}
    joints = [joints[o] for o in jorder]
    geoms = [geoms[o] for o in gorder]
    for b in bodies:
        b["joints"] = [jmap[j] for j in b["joints"]]
        b["geoms"] = [gmap[g] for g in b["geoms"]]

    nbody, njnt, ngeom = len(bodies), len(joints), len(geoms)
    m.nbody, m.njnt, m.ngeom = nbody, njnt, ngeom
    m.body_names = [b["name"] for b in bodies]
    m.jnt_names = [j["name"] for j in joints]
    m.geom_names = [g["name"] for g in geoms]
    A = m.arrays

    # ---- joints / dofs ----------------------------------------------------------
    qadr = vadr = 0
    jnt_qposadr, jnt_dofadr = [], []
    dof_body, dof_jnt, dof_parent = [], [], []
    body_last_dof = [-1] * nbody
    for bi, b in enumerate(bodies):
        last = body_last_dof[b["parent"]] if bi > 0 else -1
        for ji in b["joints"]:
            j = joints[ji]
            jnt_qposadr.append(qadr)
            jnt_dofadr.append(vadr)
            nd = 6 if j["type"] == JNT_FREE else 1
            for _ in range(nd):
                dof_body.append(bi)
                dof_jnt.append(ji)
                dof_parent.append(last)
                last = vadr
                vadr += 1
            qadr += 7 if j["type"] == JNT_FREE else 1
        body_last_dof[bi] = last
    m.nq, m.nv = qadr, vadr
    nv = m.nv

    A["body_parentid"] = np.array([b["parent"] for b in bodies], dtype=np.int32)
    rootid = np.zeros(nbody, dtype=np.int32)
    for bi in range(1, nbody):
        p = bodies[bi]["parent"]
        rootid[bi] = bi if p == 0 else rootid[p]
    A["body_rootid"] = rootid
    A["body_pos"] = np.array([b["pos"] for b in bodies])
    A["body_quat"] = np.array([b["quat"] for b in bodies])
    A["body_jntnum"] = np.array([len(b["joints"]) for b in bodies], dtype=np.int32)
    A["body_jntadr"] = np.array([b["joints"][0] if b["joints"] else -1 for b in bodies], dtype=np.int32)
    body_dofnum = np.array([sum(6 if joints[j]["type"] == JNT_FREE else 1 for j in b["joints"]) for b in bodies], dtype=np.int32)
    A["body_dofnum"] = body_dofnum
    A["body_dofadr"] = np.array([jnt_dofadr[b["joints"][0]] if b["joints"] else -1 for b in bodies], dtype=np.int32)
    A["jnt_type"] = np.array([j["type"] for j in joints], dtype=np.int32)
    A["jnt_qposadr"] = np.array(jnt_qposadr, dtype=np.int32)
    A["jnt_dofadr"] = np.array(jnt_dofadr, dtype=np.int32)
    A["jnt_bodyid"] = np.array([j["body"] for j in joints], dtype=np.int32)
    A["jnt_pos"] = np.array([j["pos"] for j in joints])
    A["jnt_axis"] = np.array([j["axis"] for j in joints])
    A["jnt_stiffness"] = np.array([j["stiffness"] for j in joints])
    A["jnt_range"] = np.array([j["range"] for j in joints])
    A["jnt_limited"] = np.array([j["limited"] for j in joints], dtype=np.int32)
    A["jnt_margin"] = np.array([j["margin"] for j in joints])
    A["jnt_solref"] = np.array([j["solref"] for j in joints])
    A["jnt_solimp"] = np.array([j["solimp"] for j in joints])
    A["dof_bodyid"] = np.array(dof_body, dtype=np.int32)
    A["dof_jntid"] = np.array(dof_jnt, dtype=np.int32)
    A["dof_parentid"] = np.array(dof_parent, dtype=np.int32)
    A["dof_armature"] = np.array([joints[j]["armature"] for j in dof_jnt])
    A["dof_damping"] = np.array([joints[j]["damping"] for j in dof_jnt])

    qpos0 = np.zeros(m.nq)
    qpos_spring = np.zeros(m.nq)
    for ji, j in enumerate(joints):
        a = jnt_qposadr[ji]
        if j["type"] == JNT_FREE:
            b = bodies[j["body"]]
            qpos0[a:a + 3] = b["pos"]
            qpos0[a + 3:a + 7] = b["quat"]
            qpos_spring[a:a + 7] = qpos0[a:a + 7]
        else:
            qpos0[a] = j["ref"]
            qpos_spring[a] = j["springref"]
    A["qpos0"], A["qpos_spring"] = qpos0, qpos_spring

    # ---- geoms ---------------------------------------------------------------
    A["geom_type"] = np.array([g["type"] for g in geoms], dtype=np.int32)
    A["geom_bodyid"] = np.array([g["body"] for g in geoms], dtype=np.int32)
    A["geom_pos"] = np.array([g["pos"] for g in geoms])
    A["geom_quat"] = np.array([g["quat"] for g in geoms])
    A["geom_size"] = np.array([g["size"] for g in geoms])

    # ---- body inertia from geoms ---------------------------------------------------
    body_mass = np.zeros(nbody)
    body_ipos = np.zeros((nbody, 3))
    body_iquat = np.tile(np.array([1.0, 0, 0, 0]), (nbody, 1))
    body_inertia = np.zeros((nbody, 3))
    for bi, b in enumerate(bodies):
        if bi == 0:
            continue
        if b["inertial"] is not None:
            it = b["inertial"]
            body_mass[bi], body_ipos[bi], body_iquat[bi], body_inertia[bi] = it["mass"], it["pos"], it["quat"], it["diag"]
            continue
        ms, cs, Is = [], [], []
        for gi in b["geoms"]:
            g = geoms[gi]
            vol, iunit = _geom_volume_inertia(g["type"], g["size"])
            mass = g["mass"] if g["mass"] is not None else g["density"] * vol
            idiag = iunit / vol * mass if vol > 0 else np.zeros(3)
            g["_mass"] = mass
            if mass <= 0:
                continue
            R = quat_to_mat(g["quat"])
            ms.append(mass)
            cs.append(g["pos"])
            Is.append(R @ np.diag(idiag) @ R.T)
        if not ms:
            continue
        M = float(np.sum(ms))
        com = np.sum([mi * ci for mi, ci in zip(ms, cs)], axis=0) / M
        I = np.zeros((3, 3))
        for mi, ci, Ii in zip(ms, cs, Is):
            d = ci - com
            I += Ii + mi * (np.dot(d, d) * np.eye(3) - np.outer(d, d))
        w, V = np.linalg.eigh(0.5 * (I + I.T))
        order = np.argsort(-w)
        w, V = w[order], V[:, order]
        if np.linalg.det(V) < 0:
            V[:, 2] = -V[:, 2]
        body_mass[bi], body_ipos[bi], body_iquat[bi], body_inertia[bi] = M, com, mat_to_quat(V), w
    A["body_mass"], A["body_ipos"], A["body_iquat"], A["body_inertia"] = body_mass, body_ipos, body_iquat, body_inertia
    # per-geom mass (explicit `mass` or density x volume; 0 where the body carries an explicit <inertial>) and friction:
    # mjModel fields the kernels never read, kept so that tests can re-derive the body constants independently
    A["geom_mass"] = np.array([g.get("_mass", 0.0) for g in geoms]).reshape(len(geoms))
    A["geom_friction"] = np.array([g["friction"] for g in geoms]).reshape(len(geoms), 3)

    # ---- actuators -----------------------------------------------------------------
    acts = []
    act_el = root.find("actuator")
    if act_el is not None:
        for el in act_el:
            if el.tag not in ("general", "motor"):
                raise NotImplementedError(f"actuator <{el.tag}>")
            attr = defaults.resolve(el, None)
            if el.tag == "motor":  # shortcut: fixed gain 1, no bias, no dynamics
                attr.update(gainprm="1", biastype="none", dyntype="none")
            gain = _floats(attr.get("gainprm", "1"))
            gear = _floats(attr.get("gear", "1"))
            ctrlrange = _floats(attr.get("ctrlrange")) if attr.get("ctrlrange") else np.zeros(2)
            cl = attr.get("ctrllimited", "auto")
            ctrllimited = (cl == "true") or (cl == "auto" and autolimits and attr.get("ctrlrange") is not None)
            forcerange = _floats(attr.get("forcerange")) if attr.get("forcerange") else np.zeros(2)
            fl = attr.get("forcelimited", "auto")
            forcelimited = (fl == "true") or (fl == "auto" and autolimits and attr.get("forcerange") is not None)
            if attr.get("biastype", "none") != "none":
                raise NotImplementedError("actuator bias (the reference deletes it, envs/rodent.py:44-45)")
            dyntype = {"none": DYN_NONE, "filter": DYN_FILTER}[attr.get("dyntype", "none")]
            dynprm = _floats(attr.get("dynprm", "1"))
            acts.append(dict(name=attr.get("name", f"act{len(acts)}"), jnt=m.jnt_names.index(attr["joint"]),
                             gain=float(gain[0]), gear=float(gear[0]), ctrlrange=ctrlrange, ctrllimited=ctrllimited,
                             forcerange=forcerange, forcelimited=forcelimited, dyntype=dyntype, dynprm=float(dynprm[0])))
    m.nu = len(acts)
    m.na = sum(1 for a in acts if a["dyntype"] != DYN_NONE)
    m.act_names = [a["name"] for a in acts]
    A["actuator_dofadr"] = np.array([jnt_dofadr[a["jnt"]] for a in acts], dtype=np.int32)
    A["actuator_gain"] = np.array([a["gain"] for a in acts])
    A["actuator_gear"] = np.array([a["gear"] for a in acts])
    A["actuator_ctrlrange"] = np.array([a["ctrlrange"] for a in acts]).reshape(-1, 2)
    A["actuator_ctrllimited"] = np.array([a["ctrllimited"] for a in acts], dtype=np.int32)
    A["actuator_forcerange"] = np.array([a["forcerange"] for a in acts]).reshape(-1, 2)
    A["actuator_forcelimited"] = np.array([a["forcelimited"] for a in acts], dtype=np.int32)
    A["actuator_dyntype"] = np.array([a["dyntype"] for a in acts], dtype=np.int32)
    A["actuator_dynprm"] = np.array([a["dynprm"] for a in acts])
    actadr, k = [], 0
    for a in acts:
        if a["dyntype"] != DYN_NONE:
            actadr.append(k)
            k += 1
        else:
            actadr.append(-1)
    A["actuator_actadr"] = np.array(actadr, dtype=np.int32)

    # ---- collision pairs -------------------------------------------------------
    pairs = _collision_pairs(root, m, bodies, geoms, defaults)
    A.update(pairs)

    # ---- constants at qpos0 ----------------------------------------------------
    _set_const(m)
    return m


def _mix_params(g1: dict, g2: dict):
    """MuJoCo contact parameter mixing (mj_contactParam / mjCPair::Compile)."""
    if g1["priority"] != g2["priority"]:
        g = g1 if g1["priority"] > g2["priority"] else g2
        condim, fr, solref, solimp = g["condim"], g["friction"], g["solref"], g["solimp"]
    else:
        condim = max(g1["condim"], g2["condim"])
        fr = np.maximum(g1["friction"], g2["friction"])
        s1, s2 = g1["solmix"], g2["solmix"]
        if s1 >= MJ_MINVAL and s2 >= MJ_MINVAL:
            mix = s1 / (s1 + s2)
        elif s1 < MJ_MINVAL and s2 < MJ_MINVAL:
            mix = 0.5
        elif s1 < MJ_MINVAL:
            mix = 0.0
        else:
            mix = 1.0
        if g1["solref"][0] > 0 and g2["solref"][0] > 0:
            solref = mix * g1["solref"] + (1 - mix) * g2["solref"]
        else:
            solref = np.minimum(g1["solref"], g2["solref"])
        solimp = mix * g1["solimp"] + (1 - mix) * g2["solimp"]
    friction5 = np.array([fr[0], fr[0], fr[1], fr[2], fr[2]])
    margin = max(g1["margin"], g2["margin"])
    gap = max(g1["gap"], g2["gap"])
    return condim, friction5, np.array(solref), np.array(solimp), margin, gap


def _collision_pairs(root, m: Model, bodies, geoms, defaults) -> Dict[str, np.ndarray]:
    """Static geom-pair list as MJX's collision driver builds it at trace time:
    explicit `<pair>`s plus contype/conaffinity candidates (same-body, parent-child with a
    non-world parent and `<exclude>`d body pairs removed).  Only plane-vs-{sphere, capsule,
    ellipsoid} functions exist on the reference path; anything else raises."""
    name2g = {g["name"]: i for i, g in enumerate(geoms)}
    name2b = {b["name"]: i for i, b in enumerate(bodies)}
    excl = set()
    out = []
    con = root.find("contact")
    if con is not None:
        for e in con.findall("exclude"):
            a, b = name2b[e.get("body1")], name2b[e.get("body2")]
            excl.add((min(a, b), max(a, b)))
        for p in con.findall("pair"):
            attr = defaults.resolve(p, None)
            g1, g2 = name2g[attr["geom1"]], name2g[attr["geom2"]]
            condim, fr5, solref, solimp, margin, gap = _mix_params(geoms[g1], geoms[g2])
            if attr.get("friction"):
                f = _floats(attr["friction"])
                fr5[: len(f)] = f
            if attr.get("solref"):
                solref = _solref(_floats(attr["solref"]))
            if attr.get("solimp"):
                solimp = _solimp(_floats(attr["solimp"]))
            if attr.get("condim"):
                condim = int(attr["condim"])
            margin = float(attr.get("margin", margin))
            gap = float(attr.get("gap", gap))
            out.append((g1, g2, condim, fr5, solref, solimp, margin - gap))
    for i in range(len(geoms)):
        for j in range(i + 1, len(geoms)):
            a, b = geoms[i], geoms[j]
            if not ((a["contype"] & b["conaffinity"]) or (b["contype"] & a["conaffinity"])):
                continue
            b1, b2 = a["body"], b["body"]
            if b1 == b2:
                continue
            # weld ids: bodies without joints are welded to their parent
            w1, w2 = _weld(bodies, b1), _weld(bodies, b2)
            if w1 == w2:
                continue
            if w1 != 0 and w2 != 0 and (_weld(bodies, bodies[w1]["parent"]) == w2 or _weld(bodies, bodies[w2]["parent"]) == w1):
                continue
            if (min(b1, b2), max(b1, b2)) in excl:
                continue
            condim, fr5, solref, solimp, margin, gap = _mix_params(a, b)
            out.append((i, j, condim, fr5, solref, solimp, margin - gap))
    rows = []
    for g1, g2, condim, fr5, solref, solimp, incl in out:
        t1, t2 = geoms[g1]["type"], geoms[g2]["type"]
        if t1 > t2:
            g1, g2, t1, t2 = g2, g1, t2, t1
        if t1 != GEOM_PLANE or t2 not in (GEOM_SPHERE, GEOM_CAPSULE, GEOM_ELLIPSOID):
            raise NotImplementedError(f"collision {t1}-{t2} is not on the reference path")
        if condim != 3:
            raise NotImplementedError("condim != 3")
        rows.append((t2, g1, g2, fr5, solref, solimp, incl))
    # MJX groups pairs by collision function; keep that grouping (sphere, capsule, ellipsoid)
    rows.sort(key=lambda r: r[0])
    n = len(rows)
    return {
        "pair_geom1": np.array([r[1] for r in rows], dtype=np.int32).reshape(n),
        "pair_geom2": np.array([r[2] for r in rows], dtype=np.int32).reshape(n),
        "pair_type": np.array([r[0] for r in rows], dtype=np.int32).reshape(n),
        "pair_friction": np.array([r[3] for r in rows]).reshape(n, 5),
        "pair_solref": np.array([r[4] for r in rows]).reshape(n, 2),
        "pair_solimp": np.array([r[5] for r in rows]).reshape(n, 5),
        "pair_includemargin": np.array([r[6] for r in rows]).reshape(n),
    }


def _weld(bodies, b: int) -> int:
    while b != 0 and not bodies[b]["joints"]:
        b = bodies[b]["parent"]
    return b


# --------------------------------------------------------------------------------------
# float64 kinematics / inertia utilities (compile-time constants, clip preprocessing)
# --------------------------------------------------------------------------------------
def kinematics(m: Model, qpos: np.ndarray):
    """FK restating `mjx.smooth.kinematics` semantics in float64 numpy.

    Returns dict(xpos, xquat, xmat, xipos, ximat, xanchor, xaxis, qpos[normalised])."""
    A = m.arrays
    nb = m.nbody
    qpos = np.array(qpos, dtype=np.float64)
    xpos = np.zeros((nb, 3))
    xquat = np.zeros((nb, 4))
    xquat[0, 0] = 1.0
    xanchor = np.zeros((m.njnt, 3))
    xaxis = np.zeros((m.njnt, 3))
    for b in range(1, nb):
        p = A["body_parentid"][b]
        pos = xpos[p] + rotate(A["body_pos"][b], xquat[p])
        quat = quat_mul(xquat[p], A["body_quat"][b])
        for k in range(A["body_jntnum"][b]):
            j = A["body_jntadr"][b] + k
            qa = A["jnt_qposadr"][j]
            if A["jnt_type"][j] == JNT_FREE:
                xanchor[j] = qpos[qa:qa + 3]
                xaxis[j] = [0, 0, 1.0]
                pos = qpos[qa:qa + 3].copy()
                quat = qpos[qa + 3:qa + 7] / np.linalg.norm(qpos[qa + 3:qa + 7])
                qpos[qa + 3:qa + 7] = quat
            else:
                anchor = rotate(A["jnt_pos"][j], quat) + pos
                axis = rotate(A["jnt_axis"][j], quat)
                xanchor[j], xaxis[j] = anchor, axis
                quat = quat_mul(quat, axis_angle_quat(A["jnt_axis"][j], qpos[qa] - A["qpos0"][qa]))
                pos = anchor - rotate(A["jnt_pos"][j], quat)
        xpos[b], xquat[b] = pos, quat
    xmat = np.array([quat_to_mat(q) for q in xquat])
    xipos = np.array([xpos[b] + xmat[b] @ A["body_ipos"][b] for b in range(nb)])
    ximat = np.array([quat_to_mat(quat_mul(xquat[b], A["body_iquat"][b])) for b in range(nb)])
    return dict(xpos=xpos, xquat=xquat, xmat=xmat, xipos=xipos, ximat=ximat, xanchor=xanchor, xaxis=xaxis, qpos=qpos)


def subtree_com(m: Model, xipos: np.ndarray) -> np.ndarray:
    A = m.arrays
    mass = A["body_mass"].copy()
    mpos = xipos * mass[:, None]
    for b in range(m.nbody - 1, 0, -1):
        p = A["body_parentid"][b]
        mass[p] += mass[b]
        mpos[p] += mpos[b]
    out = xipos.copy()
    ok = mass > MJ_MINVAL
    out[ok] = mpos[ok] / mass[ok, None]
    return out


def mass_matrix(m: Model, qpos: np.ndarray) -> np.ndarray:
    """Dense joint-space inertia via body Jacobians: M = sum_b J_b^T [m I; R I R^T] J_b + armature.
    Deliberately a different formulation from the composite-rigid-body one in oracle/ and csrc/."""
    A = m.arrays
    k = kinematics(m, qpos)
    nv = m.nv
    M = np.zeros((nv, nv))
    for b in range(1, m.nbody):
        if A["body_mass"][b] <= 0:
            continue
        jp_, jr = body_jacobian(m, k, b, k["xipos"][b])
        Iw = k["ximat"][b] @ np.diag(A["body_inertia"][b]) @ k["ximat"][b].T
        M += A["body_mass"][b] * jp_.T @ jp_ + jr.T @ Iw @ jr
    M += np.diag(A["dof_armature"])
    return M


def body_jacobian(m: Model, k: dict, body: int, point: np.ndarray):
    """(3, nv) translational and rotational Jacobians of a world point attached to `body`."""
    A = m.arrays
    jacp = np.zeros((3, m.nv))
    jacr = np.zeros((3, m.nv))
    b = body
    while b != 0:
        for kk in range(A["body_jntnum"][b]):
            j = A["body_jntadr"][b] + kk
            d = A["jnt_dofadr"][j]
            if A["jnt_type"][j] == JNT_FREE:
                jacp[:, d:d + 3] = np.eye(3)
                R = k["xmat"][b]
                for a in range(3):
                    ax = R[:, a]
                    jacr[:, d + 3 + a] = ax
                    jacp[:, d + 3 + a] = np.cross(ax, point - k["xpos"][b])
            else:
                ax = k["xaxis"][j]
                jacr[:, d] = ax
                jacp[:, d] = np.cross(ax, point - k["xanchor"][j])
        b = A["body_parentid"][b]
    return jacp, jacr


def _set_const(m: Model) -> None:
    """`mj_setConst` subset: dof_invweight0, body_invweight0, stat.meaninertia at qpos0."""
    A = m.arrays
    nv = m.nv
    if nv == 0:
        return
    M = mass_matrix(m, A["qpos0"])
    Minv = np.linalg.inv(M)
    m.meaninertia = float(np.mean(np.diag(M)))
    k = kinematics(m, A["qpos0"])
    binv = np.zeros((m.nbody, 2))
    for b in range(1, m.nbody):
        if _has_dof_ancestor(m, b):
            jp_, jr = body_jacobian(m, k, b, k["xipos"][b])
            Ap = jp_ @ Minv @ jp_.T
            Ar = jr @ Minv @ jr.T
            binv[b] = [np.trace(Ap) / 3.0, np.trace(Ar) / 3.0]
    dinv = np.diag(Minv).copy()
    for j in range(m.njnt):
        if A["jnt_type"][j] == JNT_FREE:
            d = A["jnt_dofadr"][j]
            dinv[d:d + 3] = np.mean(dinv[d:d + 3])
            dinv[d + 3:d + 6] = np.mean(dinv[d + 3:d + 6])
    A["body_invweight0"] = binv
    A["dof_invweight0"] = dinv


def _has_dof_ancestor(m: Model, b: int) -> bool:
    A = m.arrays
    while b != 0:
        if A["body_jntnum"][b] > 0:
            return True
        b = A["body_parentid"][b]
    return False


# --------------------------------------------------------------------------------------
# reference-env model recipes
# --------------------------------------------------------------------------------------
def load_rodent(mjcf_path: str, scale_factor: float = 0.9, solver: str = "cg", iterations: int = 6,
                ls_iterations: int = 6, torque: bool = True) -> Model:
    """Model exactly as `RodentTracking.__init__` builds it (`envs/rodent.py:39-63`):
    torque-actuator edit, dm_control rescale, compile, pyramidal cone, solver overrides.
    `torque=False` gives the un-edited model `process_clip` uses for kinematics
    (`mjx_preprocess.py:75-82`; actuators do not affect FK)."""
    root = load_xml(mjcf_path)
    if torque:
        torque_actuators(root)
    else:
        for a in list(root.findall("actuator")):
            root.remove(a)
    rescale_subtree(root, scale_factor, scale_factor)
    return compile_model(root, name="rodent", solver=solver, iterations=iterations, ls_iterations=ls_iterations)


def load_rodent_pair(mjcf_path: str, scale_factor: float = 0.9, solver: str = "cg", iterations: int = 6,
                     ls_iterations: int = 6) -> Model:
    """`assets/rodent_pair.xml` (two replicated rodents; render-only overlay model in the reference, `train.py:295-320`)
    compiled with the rodent env recipe (torque actuators, 0.9 rescale) for the physics-only throughput sweep of
    BASELINE.json configs[4]."""
    root = load_xml(mjcf_path)
    comp = {}
    for c in root.findall("compiler"):
        comp.update(c.attrib)
    expand_replicate(root, comp.get("angle", "degree") == "degree", comp.get("eulerseq", "xyz"))
    torque_actuators(root)
    rescale_subtree(root, scale_factor, scale_factor)
    return compile_model(root, name="rodent_pair", solver=solver, iterations=iterations, ls_iterations=ls_iterations)


def fuse_jointless_bodies(root: ET.Element) -> None:
    """brax `io.mjcf.load` fuses every body that has no joint into its parent before compiling (`_fuse_bodies`,
    reached from `envs/ant.py:40`): the body's geoms / sites / cameras / child bodies move up, their `pos` (`fromto`) and
    orientation composed with the fused body's frame, appended after the parent's remaining children.  ant.xml loses its
    four `*_leg` bodies that way (nbody 14 -> 10, SURVEY 8d config 1)."""
    comp = {}
    for c in root.findall("compiler"):
        comp.update(c.attrib)
    degree = comp.get("angle", "degree") == "degree"
    eulerseq = comp.get("eulerseq", "xyz")

    def fuse(elem: ET.Element) -> None:
        for child in list(elem):
            fuse(child)
            if child.tag != "body" or any(e.tag in ("joint", "freejoint") for e in child):
                continue
            cpos = _floats(child.get("pos")) if child.get("pos") else np.zeros(3)
            cquat = _orientation(child.attrib, degree, eulerseq)
            moved = not (np.allclose(cpos, 0.0) and np.allclose(cquat, [1.0, 0, 0, 0]))
            for g in list(child):
                if moved and g.tag in ("body", "geom", "site", "camera", "light"):
                    if g.get("fromto") is not None:
                        ft = _floats(g.get("fromto"))
                        g.set("fromto", _fmt(np.concatenate([cpos + rotate(ft[:3], cquat), cpos + rotate(ft[3:], cquat)])))
                    else:
                        gpos = _floats(g.get("pos")) if g.get("pos") else np.zeros(3)
                        gquat = _orientation(g.attrib, degree, eulerseq)
                        for k in ("euler", "axisangle", "xyaxes", "zaxis"):
                            g.attrib.pop(k, None)
                        g.set("pos", _fmt(cpos + rotate(gpos, cquat)))
                        g.set("quat", _fmt(quat_mul(cquat, gquat)))
                elem.append(g)
            elem.remove(child)

    wb = root.find("worldbody")
    if wb is not None:
        fuse(wb)


def load_ant(mjcf_path: str, solver: str = "newton", iterations: int = 1, ls_iterations: int = 4) -> Model:
    """`AntTracking.__init__` (`envs/ant.py:40-52`): brax-style load (jointless bodies fused), solver overrides from
    `configs/env_config.yaml:17-23`, eulerdamp disabled.  The `init_qpos` custom numeric (ant.xml:11) rides along as
    `arrays["init_qpos"]`: the reference's still clip is that pose tiled."""
    root = load_xml(mjcf_path)
    fuse_jointless_bodies(root)
    m = compile_model(root, name="ant", solver=solver, iterations=iterations, ls_iterations=ls_iterations, eulerdamp=False)
    for num in root.iter("numeric"):
        if num.get("name") == "init_qpos":
            m.arrays["init_qpos"] = _floats(num.get("data"))
    return m


def load_humanoid(mjcf_path: str, solver: str = "cg", iterations: int = 6, ls_iterations: int = 6) -> Model:
    """`HumanoidTracking.__init__` (`envs/humanoid.py:40-54`): no rescale, eulerdamp disabled."""
    root = load_xml(mjcf_path)
    return compile_model(root, name="humanoid", solver=solver, iterations=iterations,
                         ls_iterations=ls_iterations, eulerdamp=False)


# --------------------------------------------------------------------------------------
# (de)serialisation of a compiled model -- lets hosts without the MJCF assets (the GPU
# box has no /root/reference) rebuild the exact same tables from a small .npz
# --------------------------------------------------------------------------------------
_SCALARS = ("name", "nq", "nv", "nu", "na", "nbody", "njnt", "ngeom", "timestep", "tolerance", "ls_tolerance", "impratio",
            "solver", "iterations", "ls_iterations", "eulerdamp", "meaninertia")


def save_model(m: Model, path: str) -> None:
    out = {f"arr_{k}": v for k, v in m.arrays.items()}
    for k in _SCALARS:
        out[f"s_{k}"] = np.array(getattr(m, k))
    out["s_gravity"] = m.gravity
    for k in ("body_names", "jnt_names", "geom_names", "act_names"):
        out[f"n_{k}"] = np.array(getattr(m, k), dtype=object).astype(str)
    np.savez_compressed(path, **out)


def load_model(path: str) -> Model:
    z = np.load(path, allow_pickle=False)
    m = Model()
    for k in z.files:
        if k.startswith("arr_"):
            m.arrays[k[4:]] = z[k]
        elif k.startswith("n_"):
            setattr(m, k[2:], [str(s) for s in z[k]])
        elif k == "s_gravity":
            m.gravity = z[k]
        elif k.startswith("s_"):
            v = z[k][()]
            name = k[2:]
            if name == "name":
                m.name = str(v)
            elif name == "eulerdamp":
                m.eulerdamp = bool(v)
            elif name in ("timestep", "tolerance", "ls_tolerance", "impratio", "meaninertia"):
                setattr(m, name, float(v))
            else:
                setattr(m, name, int(v))
    return m
