"""Pins for the parts of the dynamics oracle that CAN be pinned without MuJoCo / MJX in the image (VERDICT r1, next-round
item 1; SURVEY App. I U1 / U2).  The reference's arithmetic lives in mujoco-mjx, which is not installable here, so dynamics
parity stays "unpinned" against the real thing; what is pinned here is everything that has an independent answer:

  (a) compile constants the kernel and the oracle SHARE (both consume the blob built by mjcf.py, so kernel-vs-oracle tests
      cannot see an error in them): geom volumes / inertias against numerical quadrature, the principal-axes body inertia
      against the summed geom tensors, `dof_invweight0` / `body_invweight0` / `meaninertia` against their definition
      evaluated with the ORACLE's composite-rigid-body M and cdof (a different code path from mjcf.mass_matrix), and the
      contact-parameter mixing of the rodent's floor pairs against the values written in rodent.xml;
  (b) closed forms of MuJoCo's soft-constraint model (Computation chapter: `aref = -b v - k imp r`, `R = (1 - imp) / imp *
      invweight`, pyramidal invweight, impedance curve) that pin `_kbi`, the impedance, `efc_D`, `aref`, the pyramid
      and the integrator end to end: a sphere at rest on a plane (equilibrium penetration, and the whole transient against a
      scalar recurrence of the same semi-implicit Euler step: critically damped with time constant solref[0]), a hinge
      pendulum (period), and a limited hinge pressed into its stop by gravity (equilibrium violation).
"""
import math
import xml.etree.ElementTree as ET

import numpy as np
import pytest

from conftest import pkg

mjcf = pkg("mjcf")
mb = pkg("model_blob")


# ---------------------------------------------------------------------------------------------------------------------
# (a) compile constants
# ---------------------------------------------------------------------------------------------------------------------
def _inside(gtype, size, p):
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    if gtype == mjcf.GEOM_SPHERE:
        return x * x + y * y + z * z <= size[0] ** 2
    if gtype == mjcf.GEOM_CAPSULE:
        r, h = size[0], size[1]
        zc = np.clip(z, -h, h)
        return x * x + y * y + (z - zc) ** 2 <= r * r
    if gtype == mjcf.GEOM_ELLIPSOID:
        return (x / size[0]) ** 2 + (y / size[1]) ** 2 + (z / size[2]) ** 2 <= 1.0
    if gtype == mjcf.GEOM_BOX:
        return (np.abs(x) <= size[0]) & (np.abs(y) <= size[1]) & (np.abs(z) <= size[2])
    if gtype == mjcf.GEOM_CYLINDER:
        return (x * x + y * y <= size[0] ** 2) & (np.abs(z) <= size[1])
    raise ValueError(gtype)


def _quadrature(gtype, size, n=120):
    """Midpoint-rule volume and diagonal inertia (unit density, geom frame) on an n^3 grid of the bounding box."""
    if gtype in (mjcf.GEOM_SPHERE,):
        half = np.array([size[0]] * 3)
    elif gtype == mjcf.GEOM_CAPSULE:
        half = np.array([size[0], size[0], size[1] + size[0]])
    elif gtype == mjcf.GEOM_CYLINDER:
        half = np.array([size[0], size[0], size[1]])
    else:
        half = np.array(size[:3], dtype=float)
    ax = [(np.arange(n) + 0.5) / n * 2 * h - h for h in half]
    g = np.stack(np.meshgrid(*ax, indexing="ij"), -1).reshape(-1, 3)
    inside = _inside(gtype, size, g)
    dv = np.prod(2 * half / n)
    p = g[inside]
    vol = inside.sum() * dv
    inertia = np.array([(p[:, 1] ** 2 + p[:, 2] ** 2).sum(), (p[:, 0] ** 2 + p[:, 2] ** 2).sum(), (p[:, 0] ** 2 + p[:, 1] ** 2).sum()]) * dv
    return vol, inertia


@pytest.mark.parametrize("gtype,size", [("GEOM_SPHERE", (0.03, 0, 0)), ("GEOM_CAPSULE", (0.012, 0.04, 0)), ("GEOM_CAPSULE", (0.03, 0.005, 0)),
                                        ("GEOM_ELLIPSOID", (0.02, 0.035, 0.011)), ("GEOM_BOX", (0.02, 0.03, 0.01)),
                                        ("GEOM_CYLINDER", (0.02, 0.05, 0))])
def test_geom_volume_and_inertia_against_quadrature(gtype, size):
    """mjcf._geom_volume_inertia (mjCGeom::GetVolume / SetInertia) against brute-force integration of the solid."""
    t = getattr(mjcf, gtype)
    v, i = mjcf._geom_volume_inertia(t, np.array(size, dtype=float))
    qv, qi = _quadrature(t, size)
    assert abs(v - qv) / qv < 4e-3, (v, qv)
    assert np.abs(i - qi).max() / qi.max() < 6e-3, (i, qi)


def test_body_inertia_is_the_principal_frame_of_the_summed_geom_tensors(rodent):
    """body_mass / body_ipos / body_iquat / body_inertia of every rodent body that carries mass: the full tensor
    R(iquat) diag(inertia) R^T about ipos must equal the sum over the body's geoms of their (quadrature-checked) tensors
    moved to the body COM by the parallel-axis theorem; masses add; the COM is the mass-weighted mean."""
    m = rodent["model"]
    A = m.arrays
    checked = 0
    for b in range(1, m.nbody):
        gs = [g for g in range(m.ngeom) if A["geom_bodyid"][g] == b and A["geom_mass"][g] > 0]
        if not gs or A["body_mass"][b] <= 0:
            continue
        ms = A["geom_mass"][gs]
        assert abs(ms.sum() - A["body_mass"][b]) <= 1e-12 * A["body_mass"][b], b
        coms = A["geom_pos"][gs]
        com = (ms[:, None] * coms).sum(0) / ms.sum()
        assert np.abs(com - A["body_ipos"][b]).max() < 1e-12, b
        I = np.zeros((3, 3))
        for g, mg, cg in zip(gs, ms, coms):
            v, iu = mjcf._geom_volume_inertia(int(A["geom_type"][g]), A["geom_size"][g])
            R = mjcf.quat_to_mat(A["geom_quat"][g])
            d = cg - com
            I += (mg / v) * (R @ np.diag(iu) @ R.T) + mg * (d @ d * np.eye(3) - np.outer(d, d))
        Rb = mjcf.quat_to_mat(A["body_iquat"][b])
        assert abs(np.linalg.det(Rb) - 1) < 1e-9 and abs(np.linalg.norm(A["body_iquat"][b]) - 1) < 1e-12
        got = Rb @ np.diag(A["body_inertia"][b]) @ Rb.T
        assert np.abs(got - I).max() <= 1e-9 * np.abs(I).max(), b
        assert np.all(np.diff(A["body_inertia"][b]) <= 1e-18)  # mju_eig3 orders the principal moments descending
        # a physical inertia tensor: positive, triangle inequality
        w = A["body_inertia"][b]
        assert w[2] > 0 and w[1] + w[2] >= w[0] * (1 - 1e-9)
        checked += 1
    assert checked >= 50
    assert abs(A["body_mass"].sum() - 0.186791) < 2e-6  # the whole-body mass the reference clip's COM pins (SURVEY 0.4)


def test_invweights_and_meaninertia_from_the_oracles_crb_inertia(rodent, oracle_mod):
    """mj_setConst: dof_invweight0 = diag(M^-1) (free-joint translations / rotations averaged), body_invweight0 = mean diagonal
    of the translational / rotational blocks of J M^-1 J^T at the body COM, stat.meaninertia = mean diag(M), all at qpos0.
    M and J come from the ORACLE's forward pass (composite rigid body algorithm; cdof about the subtree COM) -- not from
    mjcf.mass_matrix / body_jacobian, which produced the blob's values."""
    m = rodent["model"]
    A = m.arrays
    qpos0 = A["qpos0"].copy()
    st = dict(qpos=qpos0[None], qvel=np.zeros((1, m.nv)), act=np.zeros((1, m.na)), qacc_warmstart=np.zeros((1, m.nv)))
    d = oracle_mod.forward_dump(rodent["model_blob"], st, None, precision=64, dims=rodent["dims"])
    M = d["qM"][0]
    assert np.abs(M - M.T).max() < 1e-15
    Minv = np.linalg.inv(M)
    # the oracle reads the blob's fp32 constants, mjcf.py computed in float64: agreement to fp32 rounding of the inputs
    assert abs(M.diagonal().mean() - m.meaninertia) <= 1e-7 * m.meaninertia
    dinv = Minv.diagonal().copy()
    dinv[0:3] = dinv[0:3].mean(); dinv[3:6] = dinv[3:6].mean()
    rel = np.abs(dinv - A["dof_invweight0"]) / np.abs(dinv)
    assert rel.max() < 2e-5, rel.max()
    cdof, com, xipos = d["cdof"][0], d["subtree_com"][0][1], d["xipos"][0]
    dof_body = A["dof_bodyid"]
    parent = A["body_parentid"]
    for b in range(1, m.nbody):
        anc = set()
        bb = b
        while bb != 0:
            anc.add(bb); bb = parent[bb]
        cols = [i for i in range(m.nv) if dof_body[i] in anc]
        jr = np.zeros((3, m.nv)); jp_ = np.zeros((3, m.nv))
        for i in cols:  # spatial motion axis about the subtree COM -> point velocity at the body COM
            jr[:, i] = cdof[i, :3]
            jp_[:, i] = cdof[i, 3:] + np.cross(cdof[i, :3], xipos[b] - com)
        t = np.trace(jp_ @ Minv @ jp_.T) / 3.0
        r = np.trace(jr @ Minv @ jr.T) / 3.0
        assert abs(t - A["body_invweight0"][b][0]) <= 2e-5 * t and abs(r - A["body_invweight0"][b][1]) <= 2e-5 * r, (b, t, r, A["body_invweight0"][b])


def _xml_geom_params(root):
    """A minimal, independent resolver of MJCF geom defaults (nested <default> classes, childclass inheritance) for the three
    attributes the contact mixing reads.  Not mjcf._Defaults."""
    parent, attrs = {}, {}

    def walk(d, par):
        name = d.get("class", "main")
        parent[name] = par
        g = d.find("geom")
        attrs[name] = dict(g.attrib) if g is not None else {}
        for c in d.findall("default"):
            walk(c, name)
    walk(root.find("default"), None)

    def resolve(cls, key, default):
        while cls is not None:
            if key in attrs[cls]:
                return attrs[cls][key]
            cls = parent[cls]
        return default
    out = {}

    def body(el, childclass):
        cc = el.get("childclass", childclass)
        for g in el.findall("geom"):
            cls = g.get("class", cc or "main")
            get = lambda k, dflt: g.get(k) if g.get(k) is not None else resolve(cls, k, dflt)
            fr = [float(x) for x in get("friction", "1 0.005 0.0001").split()]
            out[g.get("name")] = dict(priority=int(get("priority", "0")), friction=fr + [1.0, 0.005, 0.0001][len(fr):],
                                      solref=[float(x) for x in get("solref", "0.02 1").split()], solmix=float(get("solmix", "1")))
        for b in el.findall("body"):
            body(b, cc)
    body(root.find("worldbody"), None)
    return out


def test_contact_parameter_mixing_of_the_rodent_floor_pairs(rodent):
    """rodent.xml:20-44: every geom inherits friction 0.7 / solref (0.005, 1); the paw classes add priority 1 and friction 1.5;
    the floor (class collision_floor) keeps priority 0.  mj_contactParam / mjCPair::Compile: the higher priority wins outright,
    equal priority -> element-wise max friction and solmix-weighted solref.  The expectation is re-derived from the XML with
    an independent default resolver and compared with the compiled pair tables the kernel and the oracle consume."""
    from conftest import reference_asset
    m = rodent["model"]
    A = m.arrays
    n = len(A["pair_geom1"])
    assert n == 32  # 27 capsules + 5 ellipsoids against the floor (SURVEY a2.4)
    assert set(A["pair_type"].tolist()) == {mjcf.GEOM_CAPSULE, mjcf.GEOM_ELLIPSOID}
    assert np.all(A["geom_type"][A["pair_geom1"]] == mjcf.GEOM_PLANE)
    fr = A["pair_friction"]
    assert np.array_equal(fr[:, 0], fr[:, 1]) and np.array_equal(fr[:, 3], fr[:, 4])  # [slide, slide, spin, roll, roll]
    # the numbers written in the file: one solref everywhere, default solimp, friction 0.7 (default) or 1.5 (paw classes)
    assert np.allclose(A["pair_solref"], [0.005, 1.0]) and np.allclose(A["pair_solimp"], [0.9, 0.95, 0.001, 0.5, 2.0])
    assert set(np.round(fr[:, 0], 9).tolist()) <= {0.7, 1.5} and np.allclose(fr[:, 2], 0.005) and np.allclose(fr[:, 3], 0.0001)
    assert np.allclose(A["pair_includemargin"], 0.0)
    path = reference_asset("rodent.xml")
    if path is None:
        pytest.skip("no VNL_REFERENCE checkout: the XML-derived expectation needs the original project's rodent.xml")
    prm = _xml_geom_params(ET.parse(path).getroot())
    npaw = 0
    for p in range(n):
        a, b = prm[m.geom_names[A["pair_geom1"][p]]], prm[m.geom_names[A["pair_geom2"][p]]]
        if a["priority"] != b["priority"]:
            w = a if a["priority"] > b["priority"] else b
            want_fr, want_sr = w["friction"], w["solref"]
            npaw += 1
        else:
            want_fr = np.maximum(a["friction"], b["friction"])
            mix = a["solmix"] / (a["solmix"] + b["solmix"])
            want_sr = mix * np.array(a["solref"]) + (1 - mix) * np.array(b["solref"])
        assert np.allclose(fr[p, [0, 2, 3]], want_fr) and np.allclose(A["pair_solref"][p], want_sr), p
        assert np.allclose(A["geom_friction"][A["pair_geom2"][p]], b["friction"])
    assert npaw == int((fr[:, 0] == 1.5).sum()) and npaw >= 4


def test_mix_params_rules():
    """mj_contactParam rules one by one on hand-made geoms: priority wins outright; equal priority -> max friction, max condim,
    solmix-weighted solref / solimp, minimum solref when one is non-positive (direct stiffness / damping form)."""
    base = dict(priority=0, condim=3, friction=np.array([1.0, 0.005, 0.0001]), solref=np.array([0.02, 1.0]),
                solimp=np.array([0.9, 0.95, 0.001, 0.5, 2.0]), solmix=1.0, margin=0.0, gap=0.0)
    g1 = dict(base, friction=np.array([0.7, 0.01, 0.0002]), solref=np.array([0.01, 1.0]), solmix=3.0, margin=0.002)
    g2 = dict(base, friction=np.array([0.9, 0.002, 0.0001]), solref=np.array([0.03, 0.5]), solmix=1.0, gap=0.001)
    condim, fr5, solref, solimp, margin, gap = mjcf._mix_params(g1, g2)
    assert condim == 3 and np.allclose(fr5, [0.9, 0.9, 0.01, 0.0002, 0.0002])
    assert np.allclose(solref, 0.75 * np.array([0.01, 1.0]) + 0.25 * np.array([0.03, 0.5])) and margin == 0.002 and gap == 0.001
    hi = dict(g2, priority=1)
    _, fr5, solref, _, _, _ = mjcf._mix_params(g1, hi)
    assert np.allclose(fr5, [0.9, 0.9, 0.002, 0.0001, 0.0001]) and np.allclose(solref, [0.03, 0.5])
    neg = dict(g2, solref=np.array([-1000.0, -10.0]))
    _, _, solref, _, _, _ = mjcf._mix_params(g1, neg)
    assert np.allclose(solref, [-1000.0, -10.0])


# ---------------------------------------------------------------------------------------------------------------------
# (b) closed forms of the soft-constraint model
# ---------------------------------------------------------------------------------------------------------------------
def _impedance(solimp, r):
    dmin, dmax, width, mid, power = solimp
    clamp = lambda v: min(max(v, 1e-4), 0.9999)  # mjMINIMP / mjMAXIMP (engine_core_constraint.c: getimpedance)
    dmin, dmax, mid, power = clamp(dmin), clamp(dmax), clamp(mid), max(1.0, power)
    x = abs(r) / width
    if x >= 1.0:
        return dmax
    y = x ** power / mid ** (power - 1) if x < mid else 1.0 - (1.0 - x) ** power / (1.0 - mid) ** (power - 1)
    return dmin + y * (dmax - dmin)


def _kb(solref, solimp, dt):
    tc, dr = max(solref[0], 2 * dt), solref[1]
    dmax = solimp[1]
    return 1.0 / (dmax * dmax * tc * tc * dr * dr), 2.0 / (dmax * tc)


def _run(oracle_mod, model, qpos, qvel, nsteps, chunks=1, precision=64, ctrl=None):
    blob = mb.build_model_blob(model)
    dims = mb.read_dims(blob)
    st = dict(qpos=np.array([qpos], dtype=np.float64), qvel=np.array([qvel], dtype=np.float64), act=np.zeros((1, model.na)),
              qacc_warmstart=np.zeros((1, model.nv)))
    traj = []
    for _ in range(chunks):
        st, _ = oracle_mod.pipeline_step(blob, st, ctrl, nsteps, precision=precision, dims=dims)
        traj.append((st["qpos"][0].copy(), st["qvel"][0].copy()))
    return traj


BALL = '''<mujoco model="ball"><option timestep="0.002"/>
<worldbody><geom name="floor" type="plane" size="5 5 .1" friction="{mu} 0.005 0.0001"/>
<body name="ball" pos="0 0 0.1"><freejoint/><geom name="g" type="sphere" size="0.05" density="{rho}" friction="{mu} 0.005 0.0001"
 solref="{tc} {dr}"/></body></worldbody></mujoco>'''


@pytest.mark.parametrize("mu,rho,tc,dr", [(1.0, 1000.0, 0.02, 1.0), (0.6, 400.0, 0.01, 1.0), (1.3, 2500.0, 0.03, 0.7)])
def test_sphere_on_plane_equilibrium_and_transient(oracle_mod, mu, rho, tc, dr):
    """A free sphere released at rest, touching the floor.  Four pyramid rows with normal Jacobian entry 1: per row
    f = D (aref - a_n),  D = imp / ((1 - imp) w),  w = (1/m)(1 + mu^2) 2 mu^2 / impratio,  aref = -b v - k imp r.
    Vertical dynamics: m a = -m g + 4 f  =>  a = (-g + c aref) / (1 + c),  c = 4 D / m.   (i) fixed point: 4 D k imp |r| = m g;
    (ii) the whole transient equals the scalar recurrence  v += dt a;  z += dt v  (semi-implicit Euler) with the impedance
    re-evaluated every step -- for mu = 1 that is the critically damped oscillator with time constant solref[0]."""
    model = mjcf.compile_model(ET.fromstring(BALL.format(mu=mu, rho=rho, tc=tc, dr=dr)), solver="cg", iterations=100, ls_iterations=50)
    A = model.arrays
    mass = A["body_mass"][1]
    assert abs(mass - rho * 4 / 3 * math.pi * 0.05 ** 3) < 1e-12 and abs(A["body_invweight0"][1][0] - 1 / mass) < 1e-9 / mass
    solimp = A["pair_solimp"][0]
    solref = 0.5 * (np.array([tc, dr]) + np.array([0.02, 1.0]))  # equal solmix: the floor's default solref mixes in
    assert np.allclose(A["pair_solref"][0], solref) and np.allclose(A["pair_friction"][0][:2], mu)
    dt, g = model.timestep, 9.81
    k, b = _kb(solref, solimp, dt)
    w = (1 / mass) * (1 + mu * mu) * 2 * mu * mu / model.impratio

    def accel(r, v):  # r = signed distance (negative in penetration)
        if r >= 0:
            return -g
        imp = _impedance(solimp, r)
        c = 4 * (imp / ((1 - imp) * w)) / mass
        a = (-g + c * (-b * v - k * imp * r)) / (1 + c)
        return a if (a - (-b * v - k * imp * r)) < 0 else -g  # rows only push

    # (ii) transient: 600 steps, compare every 20th state
    z, v = -1e-4, 0.0
    rec = []
    for i in range(600):
        v += dt * accel(z, v)
        z += dt * v
        if (i + 1) % 20 == 0:
            rec.append((z, v))
    traj = _run(oracle_mod, model, [0, 0, 0.05 - 1e-4, 1, 0, 0, 0], np.zeros(6), 20, chunks=30)
    for (qz, qv), (rz, rv) in zip(traj, rec):
        assert abs((qz[2] - 0.05) - rz) < 2e-9 and abs(qv[2] - rv) < 2e-7, ((qz[2] - 0.05, rz), (qv[2], rv))
        assert np.abs(qz[:2]).max() < 1e-12 and np.abs(qv[[0, 1, 3, 4, 5]]).max() < 1e-10  # the tangential pyramid parts cancel
    # (i) fixed point after 1.2 s (60 time constants): 4 D k imp |r| = m g with imp = imp(|r|); what is left is the solver's
    # stopping tolerance (1e-8 x meaninertia x nv on cost improvement / gradient)
    r_eq = traj[-1][0][2] - 0.05
    imp = _impedance(solimp, r_eq)
    lhs = 4 * (imp / ((1 - imp) * w)) * k * imp * abs(r_eq)
    assert r_eq < 0 and abs(lhs - mass * g) < 2e-5 * mass * g
    if mu == 1.0:  # closed form: |r| = g (1 - imp) / (k imp^2)
        assert abs(abs(r_eq) - g * (1 - imp) / (k * imp * imp)) < 2e-5 * abs(r_eq)


def test_sphere_on_plane_fp32_oracle_agrees(oracle_mod):
    """The fp32 build of the oracle (the one the GPU kernel is compared with) settles at the same penetration."""
    model = mjcf.compile_model(ET.fromstring(BALL.format(mu=1.0, rho=1000.0, tc=0.02, dr=1.0)), solver="cg", iterations=100, ls_iterations=50)
    t64 = _run(oracle_mod, model, [0, 0, 0.0499, 1, 0, 0, 0], np.zeros(6), 600)[-1][0][2]
    t32 = _run(oracle_mod, model, [0, 0, 0.0499, 1, 0, 0, 0], np.zeros(6), 600, precision=32)[-1][0][2]
    assert abs(t64 - t32) < 2e-6 and abs((t64 - 0.05) + 3.6718e-4) < 1e-7


PEND = '''<mujoco model="pend"><option timestep="0.001"><flag eulerdamp="{ed}"/></option>
<worldbody><body name="arm" pos="0 0 1"><joint name="h" type="hinge" axis="0 1 0" damping="{damp}" {limit}/>
<geom name="g" type="capsule" fromto="0 0 0 0 0 -0.4" size="0.02" density="1200"/></body></worldbody></mujoco>'''


def test_hinge_pendulum_period(oracle_mod):
    """Small oscillations of a compound pendulum: T = 2 pi sqrt(I_pivot / (m g l)).  Pins the CRB inertia, the RNE gravity
    bias and the integrator's step (semi-implicit Euler: period error O(dt^2))."""
    model = mjcf.compile_model(ET.fromstring(PEND.format(ed="disable", damp="0", limit="")), solver="cg", iterations=6, ls_iterations=6)
    A = model.arrays
    mass, l = A["body_mass"][1], abs(A["body_ipos"][1][2])
    R = mjcf.quat_to_mat(A["body_iquat"][1])
    Icom = (R @ np.diag(A["body_inertia"][1]) @ R.T)[1, 1]
    Ipiv = Icom + mass * l * l
    T = 2 * math.pi * math.sqrt(Ipiv / (mass * 9.81 * l))
    th0 = 0.01
    traj = _run(oracle_mod, model, [th0], [0.0], 1, chunks=3000)
    th = np.array([q[0] for q, _ in traj])
    t = (np.arange(len(th)) + 1) * model.timestep
    zc = [i for i in range(1, len(th)) if th[i - 1] > 0 >= th[i]]  # downward zero crossings, linearly interpolated
    tz = [t[i - 1] + (t[i] - t[i - 1]) * th[i - 1] / (th[i - 1] - th[i]) for i in zc]
    period = float(np.mean(np.diff(tz)))
    assert len(tz) >= 2 and abs(period - T) / T < 2e-4, (period, T)
    assert abs(th.max() - th0) < 2e-5 and abs(th.min() + th0) < 2e-5  # no numerical damping to first order


def test_limited_hinge_pressed_into_its_stop(oracle_mod):
    """Gravity presses the arm into the upper joint limit.  One limit row, J = -1 on the dof, invweight = dof_invweight0 = 1 / I:
    D = I imp / (1 - imp).  Rest: torque_g = D k imp |r|  =>  |r| = tau (1 - imp) / (I k imp^2), tau = m g l sin(theta)."""
    lim = math.radians(40.0)
    model = mjcf.compile_model(ET.fromstring(PEND.format(ed="enable", damp="0.002", limit='range="-20 40" limited="true"')),
                               solver="cg", iterations=50, ls_iterations=50)
    A = model.arrays
    assert abs(A["jnt_range"][0][1] - lim) < 1e-12
    mass, l = A["body_mass"][1], abs(A["body_ipos"][1][2])
    R = mjcf.quat_to_mat(A["body_iquat"][1])
    I = (R @ np.diag(A["body_inertia"][1]) @ R.T)[1, 1] + mass * l * l
    assert abs(A["dof_invweight0"][0] - 1 / I) < 1e-9 / I
    # start past the stop with the arm raised so that gravity pushes further into it: axis +y, theta > 0 swings towards -x;
    # flip gravity's lever by starting on the far side: use a tilted gravity instead (keeps the model one-liner)
    model.gravity = np.array([-9.81, 0.0, 0.0])  # pushes theta up for a downward-hanging arm
    th = _run(oracle_mod, model, [lim + 1e-3], [0.0], 4000)[-1]
    theta, vel = th[0][0], th[1][0]
    r = lim - theta
    assert r < 0 and abs(vel) < 1e-9
    solimp, solref = A["jnt_solimp"][0], A["jnt_solref"][0]
    k, _ = _kb(solref, solimp, model.timestep)
    imp = _impedance(solimp, r)
    tau = mass * 9.81 * l * math.cos(theta)  # gravity along -x on an arm hanging along -z rotated by theta about y
    want = tau * (1 - imp) / (I * k * imp * imp)
    assert abs(abs(r) - want) < 2e-4 * want, (r, want)  # what is left is the solver's stopping tolerance on a 1e-5 N m torque balance


def test_implicit_joint_damping_decay(oracle_mod):
    """forward.euler with eulerdamp (mjx euler: qacc = (M + dt diag(damping))^-1 (qfrc_smooth + qfrc_constraint), with qfrc_smooth
    carrying the passive -d v): a hinge without gravity coasts as  v' = v I / (I + dt d)  per step -- exactly, whatever dt d / I is;
    with the flag disabled it is the explicit  v' = v (1 - dt d / I).  Pins the passive damping force, the second factorisation
    (M + dt D) and its solve."""
    for ed, damp, n in (("enable", 0.02, 200), ("disable", 0.02, 200), ("enable", 5.0, 3)):  # dt d / I = 0.03, and 8 (stiff: 3 steps)
        model = mjcf.compile_model(ET.fromstring(PEND.format(ed=ed, damp=str(damp), limit="")), solver="cg", iterations=6, ls_iterations=6)
        model.gravity = np.zeros(3)
        A = model.arrays
        mass, l = A["body_mass"][1], abs(A["body_ipos"][1][2])
        R = mjcf.quat_to_mat(A["body_iquat"][1])
        I = (R @ np.diag(A["body_inertia"][1]) @ R.T)[1, 1] + mass * l * l
        dt, v0 = model.timestep, 1.5
        fac = I / (I + dt * damp) if ed == "enable" else 1.0 - dt * damp / I
        (q, v), = _run(oracle_mod, model, [0.0], [v0], n)
        # the blob stores the model constants (inertia, damping) in fp32: 6e-8 relative each, times up to n dt d / I sensitivity
        assert abs(v[0] - v0 * fac ** n) < 2e-6 * v0 * fac ** n, (ed, damp, v[0], v0 * fac ** n)
        theta = dt * v0 * fac * (1 - fac ** n) / (1 - fac)  # semi-implicit Euler: the position advances with the NEW velocity
        assert abs(q[0] - theta) < 2e-6 * abs(theta)
        (q32, v32), = _run(oracle_mod, model, [0.0], [v0], n, precision=32)
        assert abs(v32[0] - v0 * fac ** n) < 2e-5 * v0 * fac ** n


MOTOR = '''<mujoco model="motor"><option timestep="0.002"><flag eulerdamp="disable"/></option>
<worldbody><body name="arm" pos="0 0 1"><joint name="h" type="hinge" axis="0 1 0"/>
<geom name="g" type="capsule" fromto="0 0 0 0 0 -0.3" size="0.03" density="900"/></body></worldbody>
<actuator><motor name="m" joint="h" gear="{gear}" ctrllimited="true" ctrlrange="-1 1"/></actuator></mujoco>'''


def test_motor_torque_and_ctrl_clamp(oracle_mod):
    """A torque actuator on a hinge without gravity: qacc = gear clip(ctrl) / I, so v_n = n dt gear u / I and
    theta_n = dt^2 gear u / I n (n + 1) / 2.  Pins the actuator force (gain x ctrl, gear as the moment arm) and the ctrl clamp."""
    gear = 3.0
    model = mjcf.compile_model(ET.fromstring(MOTOR.format(gear=gear)), solver="cg", iterations=6, ls_iterations=6)
    model.gravity = np.zeros(3)
    A = model.arrays
    mass, l = A["body_mass"][1], abs(A["body_ipos"][1][2])
    R = mjcf.quat_to_mat(A["body_iquat"][1])
    I = (R @ np.diag(A["body_inertia"][1]) @ R.T)[1, 1] + mass * l * l
    dt, n = model.timestep, 50
    for u, ueff in ((0.4, 0.4), (-0.25, -0.25), (2.5, 1.0)):  # the last one is clamped to the ctrl range
        (q, v), = _run(oracle_mod, model, [0.0], [0.0], n, ctrl=np.array([[u]]))
        a = gear * ueff / I
        assert abs(v[0] - n * dt * a) < 2e-7 * abs(n * dt * a), (u, v[0], n * dt * a)  # fp32 constants in the blob
        assert abs(q[0] - dt * dt * a * n * (n + 1) / 2) < 2e-7 * abs(dt * dt * a * n * n)


def test_sliding_spinning_sphere_against_a_dense_qp_restatement(oracle_mod):
    """Friction.  A sphere thrown along the floor with spin: every step of the oracle (teacher-forced on its own state) against an
    independent dense statement of MuJoCo's primal problem for the one pyramidal contact,
        qacc = argmin 1/2 (a - a0)^T M (a - a0) + sum_i 1/2 D_i min(0, J_i a - aref_i)^2 ,   a0 = M^-1 qfrc_smooth = gravity,
    solved here by an exact active-set Newton iteration on the 6 x 6 system (numpy, float64).  Rows: J_i = d_i^T [I | -[r]x R] with
    d_i = n +- mu t_k (k = 1, 2), r = contact point - centre, contact point = centre - n (radius + dist / 2), free-joint angular
    velocity in the BODY frame (hence R); aref_i = -b J_i v - k imp dist, D = imp / ((1 - imp) w), w = (1/m)(1 + mu^2) 2 mu^2 / impratio.
    Pins the pyramid directions, the contact point, the rotational block of the contact Jacobian and the solver's convergence with
    friction rows active (sliding, then rolling)."""
    mu, rho, rad = 0.7, 800.0, 0.05
    model = mjcf.compile_model(ET.fromstring(BALL.format(mu=mu, rho=rho, tc=0.02, dr=1.0)), solver="cg", iterations=200, ls_iterations=50)
    A = model.arrays
    mass = A["body_mass"][1]
    Ib = A["body_inertia"][1]
    assert np.allclose(Ib, 0.4 * mass * rad * rad, rtol=1e-6)  # solid sphere
    M = np.diag([mass] * 3 + list(Ib))
    solimp, solref = A["pair_solimp"][0], A["pair_solref"][0]
    dt, g = model.timestep, 9.81
    k, b = _kb(solref, solimp, dt)
    w = (1 / mass) * (1 + mu * mu) * 2 * mu * mu / model.impratio
    n = np.array([0.0, 0.0, 1.0])
    tang = (np.array([1.0, 0.0, 0.0]), np.array([0.0, 1.0, 0.0]))  # any orthonormal pair: the set {n +- mu t_k} decides, not the order

    def skew(v):
        return np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])

    def qp(qpos, qvel):
        dist = qpos[2] - rad
        a0 = np.array([0, 0, -g, 0, 0, 0.0])  # no bias torque: isotropic inertia, omega x I omega = 0
        if dist >= 0:
            return a0
        R = mjcf.quat_to_mat(qpos[3:7])
        r = -n * (rad + 0.5 * dist)
        Jp = np.hstack([np.eye(3), -skew(r) @ R])
        J = np.array([(n + sgn * mu * t) @ Jp for t in tang for sgn in (1.0, -1.0)])
        imp = _impedance(solimp, dist)
        D = imp / ((1 - imp) * w)
        aref = -b * (J @ qvel) - k * imp * dist
        act = np.ones(4, bool)
        for _ in range(20):  # active-set Newton: exact for a piecewise-quadratic convex objective once the set is right
            Ja = J[act]
            a = np.linalg.solve(M + D * Ja.T @ Ja, M @ a0 + D * Ja.T @ aref[act])
            new = (J @ a - aref) < 0
            if (new == act).all():
                return a
            act = new
        raise AssertionError("active set did not settle")

    qpos = np.array([0, 0, rad - 3.0e-4, 1, 0, 0, 0.0])
    qvel = np.array([0.6, -0.2, 0.0, 3.0, 5.0, -2.0])  # sliding along x / -y with spin about all axes (body frame)
    blob = mb.build_model_blob(model)
    dims = mb.read_dims(blob)
    st = dict(qpos=qpos[None].copy(), qvel=qvel[None].copy(), act=np.zeros((1, 0)), qacc_warmstart=np.zeros((1, 6)))
    worst, slid, rolled, errs = 0.0, False, False, []
    for step in range(400):
        want = st["qvel"][0] + dt * qp(st["qpos"][0], st["qvel"][0])
        R = mjcf.quat_to_mat(st["qpos"][0][3:7])
        vslip = st["qvel"][0][:3] + np.cross(R @ st["qvel"][0][3:], -n * rad)
        slid |= float(np.hypot(vslip[0], vslip[1])) > 0.1
        rolled |= step > 50 and float(np.hypot(vslip[0], vslip[1])) < 1e-3
        st, _ = oracle_mod.pipeline_step(blob, st, None, 1, precision=64, dims=dims)
        err = float(np.abs(st["qvel"][0] - want).max())
        worst = max(worst, err)
        errs.append(err)
    assert slid and rolled  # the run covers the sliding phase and the rolling one
    # typical agreement 1e-8 (fp32 model constants in the blob); the worst steps are the first ones of the sliding phase, where the
    # friction torque on the tiny inertia gives angular accelerations of ~350 rad/s^2 and the CG solver's stopping rule
    # (improvement / gradient < 1e-8 x meaninertia x nv) leaves 1e-6 rad/s per step
    assert float(np.median(errs)) < 5e-8 and worst < 5e-6, (float(np.median(errs)), worst)


REST = '''<mujoco model="rest"><option timestep="0.002"/>
<worldbody><geom name="floor" type="plane" size="5 5 .1"/>
<body name="b" pos="0 0 {z}" {quat}><freejoint/><geom name="g" {geom} density="700"/></body></worldbody></mujoco>'''


@pytest.mark.parametrize("geom,bottom,ncon,quat", [
    ('type="capsule" fromto="-0.08 0 0 0.08 0 0" size="0.03"', 0.03, 2, ""),               # lying flat: one contact under each end sphere
    ('type="ellipsoid" size="0.08 0.05 0.03"', 0.03, 1, ""),                                # support point under the centre
    ('type="ellipsoid" size="0.03 0.05 0.08"', 0.05, 1, 'quat="0.5 0.5 0.5 0.5"'),          # 120 deg about (1, 1, 1): local y (0.05) is vertical
])
def test_capsule_and_ellipsoid_rest_on_the_plane(oracle_mod, geom, bottom, ncon, quat):
    """The other two plane colliders of the rodent (plane_capsule: two plane-sphere tests at the end spheres; plane_ellipsoid: support
    point along -normal in the geom frame).  At rest every contact carries 4 pyramid rows of the same D:
    (4 ncon) D k imp |r| = m g  with the sphere test's D and w -- which holds only if the colliders report the right distance for
    the right number of contacts, and the body does not tip (contact points symmetric about the COM)."""
    mu = 1.0
    z0 = bottom - 2e-4
    model = mjcf.compile_model(ET.fromstring(REST.format(z=z0, geom=geom, quat=quat)), solver="cg", iterations=100, ls_iterations=50)
    A = model.arrays
    mass = A["body_mass"][1]
    solimp, solref = A["pair_solimp"][0], A["pair_solref"][0]
    assert np.allclose(A["pair_friction"][0][:2], mu)
    k, _ = _kb(solref, solimp, model.timestep)
    w = A["body_invweight0"][1][0] * (1 + mu * mu) * 2 * mu * mu / model.impratio
    assert abs(A["body_invweight0"][1][0] - 1 / mass) < 1e-6 / mass  # translational inverse weight of a free body
    q0 = A["qpos0"].copy()
    (q, v), = _run(oracle_mod, model, q0, np.zeros(6), 800)
    r = q[2] - bottom
    imp = _impedance(solimp, r)
    lhs = 4 * ncon * (imp / ((1 - imp) * w)) * k * imp * abs(r)
    assert r < 0 and abs(lhs - mass * 9.81) < 1e-4 * mass * 9.81, (r, lhs, mass * 9.81)
    assert np.abs(v).max() < 5e-6 and np.abs(q[:2]).max() < 1e-6  # at rest (to the solver's stopping tolerance), not sliding
    assert np.abs(q[3:7] - q0[3:7]).max() < 1e-6  # and not tipping


DPEND = '''<mujoco model="dpend"><option timestep="0.001"/>
<worldbody><body name="l1" pos="0 0 1"><joint name="h1" type="hinge" axis="0 1 0"/>
<geom name="g1" type="capsule" fromto="0 0 0 0 0 -0.3" size="0.02" density="1100"/>
<body name="l2" pos="0 0 -0.3"><joint name="h2" type="hinge" axis="0 1 0"/>
<geom name="g2" type="capsule" fromto="0 0 0 0 0 -0.22" size="0.015" density="900"/></body></body></worldbody></mujoco>'''


def test_double_pendulum_inertia_and_bias_against_the_lagrangian(oracle_mod):
    """A planar double pendulum: the oracle's composite-rigid-body M(q) and recursive-Newton-Euler bias c(q, v) + g(q) against the
    textbook Lagrangian
        M11 = m1 lc1^2 + I1 + m2 (l1^2 + lc2^2 + 2 l1 lc2 cos q2) + I2,  M12 = m2 (lc2^2 + l1 lc2 cos q2) + I2,  M22 = m2 lc2^2 + I2,
        c = h (-(2 v1 v2 + v2^2), v1^2),  h = m2 l1 lc2 sin q2,
        g = (m1 g lc1 sin q1 + m2 g (l1 sin q1 + lc2 sin(q1 + q2)),  m2 g lc2 sin(q1 + q2)).
    Pins the chain part of kinematics / com / cdof / CRB / RNE (Coriolis and centrifugal terms included) without reference to any
    of the repo's own inertia code; then 300 steps of the oracle against semi-implicit Euler on these equations of motion."""
    model = mjcf.compile_model(ET.fromstring(DPEND), solver="cg", iterations=6, ls_iterations=6)
    A = model.arrays
    blob = mb.build_model_blob(model)
    dims = mb.read_dims(blob)
    m1, m2 = A["body_mass"][1], A["body_mass"][2]
    lc1, lc2, l1 = abs(A["body_ipos"][1][2]), abs(A["body_ipos"][2][2]), 0.3
    Iy = lambda b: (mjcf.quat_to_mat(A["body_iquat"][b]) @ np.diag(A["body_inertia"][b]) @ mjcf.quat_to_mat(A["body_iquat"][b]).T)[1, 1]
    I1, I2, g = Iy(1), Iy(2), 9.81

    def lagr(q, v):
        c2, s2 = math.cos(q[1]), math.sin(q[1])
        M = np.array([[m1 * lc1 ** 2 + I1 + m2 * (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * c2) + I2, m2 * (lc2 ** 2 + l1 * lc2 * c2) + I2],
                      [m2 * (lc2 ** 2 + l1 * lc2 * c2) + I2, m2 * lc2 ** 2 + I2]])
        h = m2 * l1 * lc2 * s2
        bias = np.array([-h * (2 * v[0] * v[1] + v[1] ** 2), h * v[0] ** 2])
        bias += np.array([m1 * g * lc1 * math.sin(q[0]) + m2 * g * (l1 * math.sin(q[0]) + lc2 * math.sin(q[0] + q[1])),
                          m2 * g * lc2 * math.sin(q[0] + q[1])])
        V = -m1 * g * lc1 * math.cos(q[0]) - m2 * g * (l1 * math.cos(q[0]) + lc2 * math.cos(q[0] + q[1]))
        return M, bias, 0.5 * v @ M @ v + V

    rng = np.random.default_rng(4)
    for _ in range(6):
        q, v = rng.uniform(-2.5, 2.5, 2), rng.uniform(-6, 6, 2)
        st = dict(qpos=q[None], qvel=v[None], act=np.zeros((1, 0)), qacc_warmstart=np.zeros((1, 2)))
        d = oracle_mod.forward_dump(blob, st, None, precision=64, dims=dims)
        M, bias, _ = lagr(q, v)
        assert np.abs(d["qM"][0] - M).max() < 1e-6 * np.abs(M).max(), (d["qM"][0], M)  # fp32 model constants in the blob
        assert np.abs(d["qfrc_bias"][0] - bias).max() < 1e-6 * max(1.0, np.abs(bias).max()), (d["qfrc_bias"][0], bias)
    # one step = semi-implicit Euler on these equations of motion: v' = v + dt M^-1 (-bias), q' = q + dt v'  (no damping, no constraints);
    # 300 steps, each predicted from the oracle's own previous state
    st = dict(qpos=np.array([[1.2, -0.7]]), qvel=np.array([[0.5, 2.0]]), act=np.zeros((1, 0)), qacc_warmstart=np.zeros((1, 2)))
    dt = model.timestep
    for _ in range(300):
        q, v = st["qpos"][0].copy(), st["qvel"][0].copy()
        M, bias, _ = lagr(q, v)
        v1 = v + dt * np.linalg.solve(M, -bias)
        st, _ = oracle_mod.pipeline_step(blob, st, None, 1, precision=64, dims=dims)
        assert np.abs(st["qvel"][0] - v1).max() < 1e-7 * max(1.0, np.abs(v1).max()) and np.abs(st["qpos"][0] - (q + dt * v1)).max() < 1e-9


TUMBLE = '''<mujoco model="tumble"><option timestep="0.002"/>
<worldbody><body name="b" pos="0 0 1"><freejoint/><geom name="g" type="ellipsoid" size="0.08 0.05 0.03" density="800"/></body></worldbody></mujoco>'''


def test_free_body_tumbles_by_eulers_equations(oracle_mod):
    """A free asymmetric body: angular velocity in the BODY frame obeys I w' = -(w x I w) (the gyroscopic part of the RNE bias),
    the quaternion advances by q <- q * exp(dt w_new) (mju_quatIntegrate: right-multiplication by the body-frame rotation), the COM
    falls with g.  Step by step against semi-implicit Euler on these equations; pins the free joint's rotational dofs end to end."""
    model = mjcf.compile_model(ET.fromstring(TUMBLE), solver="cg", iterations=6, ls_iterations=6)
    A = model.arrays
    blob = mb.build_model_blob(model)
    dims = mb.read_dims(blob)
    Ri = mjcf.quat_to_mat(A["body_iquat"][1])
    Ib = Ri @ np.diag(A["body_inertia"][1]) @ Ri.T  # inertia in the body frame (the compiler sorts the principal moments)
    mass = A["body_mass"][1]
    want = mass / 5 * np.array([0.05 ** 2 + 0.03 ** 2, 0.08 ** 2 + 0.03 ** 2, 0.08 ** 2 + 0.05 ** 2])  # solid ellipsoid
    assert np.abs(Ib - np.diag(want)).max() < 1e-9 * want.max() and np.abs(A["body_ipos"][1]).max() < 1e-15
    dt, g = model.timestep, np.array([0, 0, -9.81])

    def quat_exp(w, h):
        a = np.linalg.norm(w) * h
        ax = w / max(np.linalg.norm(w), 1e-300)
        return np.concatenate([[math.cos(a / 2)], math.sin(a / 2) * ax])

    st = dict(qpos=np.array([[0.1, -0.2, 1.0, 0.8, 0.2, -0.4, 0.4]]), qvel=np.array([[0.3, 0.1, -0.2, 3.0, -2.0, 5.0]]), act=np.zeros((1, 0)),
              qacc_warmstart=np.zeros((1, 6)))
    st["qpos"][0, 3:7] /= np.linalg.norm(st["qpos"][0, 3:7])
    for _ in range(300):
        q, v = st["qpos"][0].copy(), st["qvel"][0].copy()
        w = v[3:]
        w1 = w + dt * np.linalg.solve(Ib, -np.cross(w, Ib @ w))
        vl1 = v[:3] + dt * g
        q1 = mjcf.quat_mul(q[3:7], quat_exp(w1, dt))
        q1 /= np.linalg.norm(q1)
        st, _ = oracle_mod.pipeline_step(blob, st, None, 1, precision=64, dims=dims)
        assert np.abs(st["qvel"][0][3:] - w1).max() < 1e-6 * np.abs(w1).max(), (st["qvel"][0][3:], w1)  # fp32 inertia constants in the blob
        assert np.abs(st["qvel"][0][:3] - vl1).max() < 1e-8 and np.abs(st["qpos"][0][:3] - (q[:3] + dt * vl1)).max() < 1e-9  # g, dt are fp32 in the blob
        assert np.abs(st["qpos"][0][3:7] - q1).max() < 1e-8, (st["qpos"][0][3:7], q1)


SPRING = '''<mujoco model="spring"><option timestep="0.001"><flag eulerdamp="disable"/></option>
<worldbody><body name="arm" pos="0 0 1"><joint name="h" type="hinge" axis="0 1 0" stiffness="{k}" springref="{ref}" armature="{arm}"/>
<geom name="g" type="capsule" fromto="0 0 0 0 0 -0.3" size="0.03" density="900"/></body></worldbody>
<actuator><general name="m" joint="h" gear="{gear}" gainprm="{gain}" dyntype="filter" dynprm="{tau}" ctrllimited="true" ctrlrange="-1 1"
 forcelimited="true" forcerange="-{fmax} {fmax}"/></actuator></mujoco>'''


def test_joint_spring_armature_and_filtered_actuator(oracle_mod):
    """(i) A hinge spring without gravity oscillates with omega^2 = k / (I + armature) about springref (semi-implicit Euler: exactly the
    recurrence v += dt (-k (q - ref)) / (I + armature), q += dt v).  (ii) A first-order activation filter act' = (ctrl - act) / tau
    drives force = clip(gain act, forcerange) through the gear; the force of a step uses the activation BEFORE its update.
    Pins jnt_stiffness / qpos_spring, dof_armature in M, actuator dynamics, gain, force clamp."""
    k, ref, arm, gear, gain, tau, fmax = 0.8, 15.0, 0.003, 2.0, 4.0, 0.05, 3.0
    model = mjcf.compile_model(ET.fromstring(SPRING.format(k=k, ref=ref, arm=arm, gear=gear, gain=gain, tau=tau, fmax=fmax)), solver="cg",
                               iterations=6, ls_iterations=6)
    model.gravity = np.zeros(3)
    A = model.arrays
    mass, l = A["body_mass"][1], abs(A["body_ipos"][1][2])
    R = mjcf.quat_to_mat(A["body_iquat"][1])
    I = (R @ np.diag(A["body_inertia"][1]) @ R.T)[1, 1] + mass * l * l + arm
    dt, qref = model.timestep, math.radians(ref)
    blob = mb.build_model_blob(model)
    dims = mb.read_dims(blob)
    assert model.na == 1 and abs(A["qpos_spring"][0] - qref) < 1e-12
    # (i) spring, actuator idle
    q, v = 0.0, 0.0
    st = dict(qpos=np.array([[q]]), qvel=np.array([[v]]), act=np.zeros((1, 1)), qacc_warmstart=np.zeros((1, 1)))
    st, _ = oracle_mod.pipeline_step(blob, st, np.zeros((1, 1)), 700, precision=64, dims=dims)
    for _ in range(700):
        v += dt * (-k * (q - qref)) / I
        q += dt * v
    assert abs(st["qpos"][0, 0] - q) < 2e-6 * abs(qref) and abs(st["qvel"][0, 0] - v) < 2e-6 * math.sqrt(k / I) * abs(qref)
    assert abs(st["qpos"][0, 0] - qref) <= abs(qref) * 1.001  # it swings about the reference angle
    # (ii) filtered actuator against the scalar recurrence, spring switched off by starting at the reference with k-force cancelling
    for u in (0.3, 1.0, -2.0):  # 1.0 saturates the force range (gain x act -> 4 > 3), -2.0 is clamped to -1 first
        ue = min(max(u, -1.0), 1.0)
        q, v, act = qref, 0.0, 0.0
        st = dict(qpos=np.array([[q]]), qvel=np.array([[v]]), act=np.zeros((1, 1)), qacc_warmstart=np.zeros((1, 1)))
        st, _ = oracle_mod.pipeline_step(blob, st, np.array([[u]]), 300, precision=64, dims=dims)
        for _ in range(300):
            force = min(max(gain * act, -fmax), fmax)
            v += dt * (gear * force - k * (q - qref)) / I
            q += dt * v
            act += dt * (ue - act) / tau
        assert abs(st["act"][0, 0] - act) < 1e-6 * abs(ue), (u, st["act"][0, 0], act)
        assert abs(st["qvel"][0, 0] - v) < 2e-6 * max(1.0, abs(v)) and abs(st["qpos"][0, 0] - q) < 2e-6 * max(1.0, abs(q)), (u, st["qvel"][0, 0], v)


def test_cg_and_newton_agree_on_the_rodent_in_contact(rodent, oracle_mod):
    """Two solvers, one convex problem: run to convergence, the oracle's CG path (M^-1-preconditioned Polak-Ribiere) and its Newton path
    (dense H = M + J^T D J, Cholesky) must give the same constrained acceleration for the rodent pressed into the floor with joint
    limits active -- two independent code paths of the restatement checking each other on the real model (303 rows, 73 dofs);
    and the result does not depend on the warm start (it only picks the starting point)."""
    import copy
    from conftest import start_states
    B = 4
    qpos, qvel, _ = start_states(rodent, B, seed=3)
    qpos = qpos.astype(np.float64); qvel = qvel.astype(np.float64)
    qpos[:, 2] -= 0.012  # into the floor: several active contacts per env
    rng = np.random.default_rng(8)
    ctrl = rng.uniform(-0.5, 0.5, size=(B, 30))
    outs = {}
    for name, solver, iters, warm in (("cg", 1, 300, 0.0), ("newton", 2, 60, 0.0), ("cg_warm", 1, 300, 1.0)):
        m = copy.copy(rodent["model"])
        m.solver, m.iterations, m.ls_iterations, m.tolerance = solver, iters, 50, 1e-12
        blob = mb.build_model_blob(m)
        dims = mb.read_dims(blob)
        st = dict(qpos=qpos.copy(), qvel=qvel.copy(), act=np.zeros((B, 30)), qacc_warmstart=warm * 50.0 * rng.standard_normal((B, 73)))
        d = oracle_mod.forward_dump(blob, st, ctrl, precision=64, dims=dims)
        outs[name] = d
        assert (d["counters"][:, 2] >= 3).all() and (d["counters"][:, 3] >= 1).all()  # contacts and limit rows active
    scale = np.abs(outs["newton"]["qacc"]).max()
    for other in ("cg", "cg_warm"):
        err = np.abs(outs[other]["qacc"] - outs["newton"]["qacc"]).max() / scale
        assert err < 1e-6, (other, err)
        ferr = np.abs(outs[other]["qfrc_constraint"] - outs["newton"]["qfrc_constraint"]).max() / np.abs(outs["newton"]["qfrc_constraint"]).max()
        assert ferr < 1e-6, (other, ferr)


def test_contact_jacobian_rows_are_the_derivative_of_the_forward_kinematics(rodent, oracle_mod):
    """efc_J of the pyramidal contact rows against central finite differences of the oracle's own forward kinematics (xpos / xmat --
    which the reference's clip golden pins, tests/test_mjcf_clip.py): for dof i, move the configuration by +-eps along the dof (free
    joint: world translation, body-frame rotation; hinges: angle), follow the material point of the contact body that sits at the
    contact position, and project its displacement on n +- mu t_k.  Also: limit rows are -+1 on their dof, and the rows' reference
    acceleration obeys aref = -b (J v) - k imp pos with (k, b, imp) from the pair's solref / solimp."""
    from conftest import start_states
    m = rodent["model"]
    A = m.arrays
    qpos, qvel, _ = start_states(rodent, 1, seed=5)
    qpos = qpos.astype(np.float64); qvel = 0.3 * qvel.astype(np.float64)
    qpos[:, 2] -= 0.012
    blob, dims = rodent["model_blob"], rodent["dims"]
    fd = lambda q: oracle_mod.forward_dump(blob, dict(qpos=q, qvel=qvel, act=np.zeros((1, 30)), qacc_warmstart=np.zeros((1, 73))), None,
                                           precision=64, dims=dims)
    d = fd(qpos)
    J, dist = d["efc_J"][0], d["con_dist"][0]
    nl = dims["nlimit"]
    act_con = [c for c in range(dims["ncon"]) if dist[c] < 0]
    assert len(act_con) >= 3

    def moved(q, i, eps):
        q = q.copy()
        if i < 3:
            q[0, i] += eps
        elif i < 6:
            w = np.zeros(3); w[i - 3] = eps
            dq = np.concatenate([[math.cos(eps / 2)], math.sin(eps / 2) * w / eps])
            q[0, 3:7] = mjcf.quat_mul(q[0, 3:7], dq)
        else:
            q[0, 7 + (i - 6)] += eps
        return q

    # contact -> (pair, body): contacts are enumerated pair by pair, a plane-capsule pair (type 3) spawns two
    pair_of = []
    for p_, t_ in enumerate(A["pair_type"]):
        pair_of += [p_] * (2 if t_ == 3 else 1)
    assert len(pair_of) == dims["ncon"]
    eps = 1e-6
    Jp = {c: np.zeros((3, 73)) for c in act_con}
    body_of = {c: int(A["geom_bodyid"][A["pair_geom2"][pair_of[c]]]) for c in act_con}
    for i in range(73):
        dp, dm = fd(moved(qpos, i, eps)), fd(moved(qpos, i, -eps))
        for c in act_con:
            b, p = body_of[c], d["con_pos"][0][c]
            loc = d["xmat"][0][b].reshape(3, 3).T @ (p - d["xpos"][0][b])
            pp = dp["xpos"][0][b] + dp["xmat"][0][b].reshape(3, 3) @ loc
            pm = dm["xpos"][0][b] + dm["xmat"][0][b].reshape(3, 3) @ loc
            Jp[c][:, i] = (pp - pm) / (2 * eps)
    checked = 0
    for c in act_con:
        fr = d["con_frame"][0][c].reshape(3, 3)
        mu = A["pair_friction"][pair_of[c]][0]
        want = [(fr[0] + sgn * mu * fr[k]) @ Jp[c] for k in (1, 2) for sgn in (1.0, -1.0)]
        rows = J[nl + 4 * c: nl + 4 * c + 4]
        assert np.abs(rows).max() > 0
        for r in rows:  # each dumped row is one of the four pyramid directions (order not assumed)
            err = min(np.abs(r - w).max() for w in want)
            assert err < 2e-6 * max(1.0, np.abs(r).max()), (c, err)
            checked += 1
    assert checked == 4 * len(act_con)
    # limit rows: one-hot on their dof; all rows: aref = -b J v - k imp pos
    pos, aref = d["efc_pos"][0], d["efc_aref"][0]
    for r in range(nl):
        if np.abs(J[r]).max() > 0:
            assert np.count_nonzero(J[r]) == 1 and abs(abs(J[r]).max() - 1.0) < 1e-12
    for c in act_con:
        k, b_ = _kb(A["pair_solref"][pair_of[c]], A["pair_solimp"][pair_of[c]], m.timestep)
        imp = _impedance(A["pair_solimp"][pair_of[c]], dist[c])
        mu_c = A["pair_friction"][pair_of[c]][0]
        w_c = A["body_invweight0"][body_of[c]][0] * (1 + mu_c * mu_c) * 2 * mu_c * mu_c / m.impratio  # the plane's body (world) adds 0
        for r in range(nl + 4 * c, nl + 4 * c + 4):
            assert abs(pos[r] - dist[c]) < 1e-12
            assert abs(d["efc_D"][0][r] - imp / ((1 - imp) * w_c)) < 1e-6 * d["efc_D"][0][r], (r, d["efc_D"][0][r], imp / ((1 - imp) * w_c))
            assert abs(aref[r] - (-b_ * (J[r] @ qvel[0]) - k * imp * dist[c])) < 1e-6 * max(1.0, abs(aref[r])), (r, aref[r])


def test_rodent_inertia_matrix_from_finite_differences_of_the_kinematics(rodent, oracle_mod):
    """M(q) = sum_b J_b^T diag(m_b 1, R_b I_b R_b^T) J_b + armature with every body Jacobian taken by central finite differences of the
    oracle's forward kinematics (xipos / ximat) -- against the oracle's composite-rigid-body qM.  The kinematics are pinned by the
    reference clip, the body inertias by quadrature (above): this closes the chain to the full 73 x 73 inertia of the rodent without
    any analytic Jacobian code in the loop."""
    from conftest import start_states
    m = rodent["model"]
    A = m.arrays
    qpos, qvel, _ = start_states(rodent, 1, seed=9)
    qpos = qpos.astype(np.float64); qvel = qvel.astype(np.float64)
    blob, dims = rodent["model_blob"], rodent["dims"]
    nb = dims["nbody"]
    fd = lambda q: oracle_mod.forward_dump(blob, dict(qpos=q, qvel=qvel, act=np.zeros((1, 30)), qacc_warmstart=np.zeros((1, 73))), None,
                                           precision=64, dims=dims)

    def moved(q, i, eps):
        q = q.copy()
        if i < 3:
            q[0, i] += eps
        elif i < 6:
            w = np.zeros(3); w[i - 3] = 1.0
            q[0, 3:7] = mjcf.quat_mul(q[0, 3:7], np.concatenate([[math.cos(eps / 2)], math.sin(eps / 2) * w]))
        else:
            q[0, 7 + (i - 6)] += eps
        return q

    d = fd(qpos)
    eps = 1e-6
    Jl, Jr = np.zeros((nb, 3, 73)), np.zeros((nb, 3, 73))
    for i in range(73):
        dp, dm = fd(moved(qpos, i, eps)), fd(moved(qpos, i, -eps))
        Jl[:, :, i] = (dp["xipos"][0] - dm["xipos"][0]) / (2 * eps)
        Rp, Rm, R0 = dp["ximat"][0].reshape(nb, 3, 3), dm["ximat"][0].reshape(nb, 3, 3), d["ximat"][0].reshape(nb, 3, 3)
        S = np.einsum("bij,bkj->bik", (Rp - Rm) / (2 * eps), R0)  # dR R^T = [w]x
        Jr[:, 0, i], Jr[:, 1, i], Jr[:, 2, i] = S[:, 2, 1], S[:, 0, 2], S[:, 1, 0]
    M = np.diag(A["dof_armature"].astype(np.float64))
    R0 = d["ximat"][0].reshape(nb, 3, 3)
    for b in range(1, nb):
        Iw = R0[b] @ np.diag(A["body_inertia"][b]) @ R0[b].T
        M += A["body_mass"][b] * Jl[b].T @ Jl[b] + Jr[b].T @ Iw @ Jr[b]
    got = d["qM"][0]
    assert np.abs(got - M).max() < 2e-6 * np.abs(M).max(), np.abs(got - M).max() / np.abs(M).max()
    assert np.linalg.eigvalsh(got).min() > 0


def test_rodent_bias_forces_balance_the_energy_rate(rodent, oracle_mod):
    """Power balance of the conservative part of the dynamics, valid in any (quasi-)velocity coordinates:
    v . qfrc_bias = 1/2 v^T (dM/dt) v + dV/dt  along the motion (from d/dt (1/2 v^T M v + V) = 0 with M v' = -bias), with dM/dt and
    dV/dt by central differences of the oracle's qM (pinned above) and of V = sum_b m_b g z_b (FK) at q integrated by +-eps v.
    Pins the power of the recursive-Newton-Euler bias (Coriolis, centrifugal, gyroscopic, gravity) on the full rodent."""
    from conftest import start_states
    m = rodent["model"]
    A = m.arrays
    blob, dims = rodent["model_blob"], rodent["dims"]
    mass = A["body_mass"].astype(np.float64)
    rng = np.random.default_rng(12)
    for trial in range(4):
        qpos, _, _ = start_states(rodent, 1, seed=20 + trial)
        qpos = qpos.astype(np.float64)
        v = np.concatenate([rng.uniform(-1, 1, 3), rng.uniform(-4, 4, 3), rng.uniform(-6, 6, 67)])
        fd = lambda q: oracle_mod.forward_dump(blob, dict(qpos=q, qvel=v[None], act=np.zeros((1, 30)), qacc_warmstart=np.zeros((1, 73))), None,
                                               precision=64, dims=dims)

        def along(q, h):
            q = q.copy()
            q[0, :3] += h * v[:3]
            a = np.linalg.norm(v[3:6]) * h
            dq = np.concatenate([[math.cos(a / 2)], math.sin(a / 2) * v[3:6] / np.linalg.norm(v[3:6])])
            q[0, 3:7] = mjcf.quat_mul(q[0, 3:7], dq)
            q[0, 7:] += h * v[6:]
            return q

        d0 = fd(qpos)
        eps = 1e-5
        dp, dm = fd(along(qpos, eps)), fd(along(qpos, -eps))
        Mdot = (dp["qM"][0] - dm["qM"][0]) / (2 * eps)
        V = lambda d: 9.81 * float(mass @ d["xipos"][0][:, 2])
        rhs = 0.5 * v @ Mdot @ v + (V(dp) - V(dm)) / (2 * eps)
        lhs = float(v @ d0["qfrc_bias"][0])
        scale = abs(0.5 * v @ Mdot @ v) + abs((V(dp) - V(dm)) / (2 * eps)) + 1e-9
        assert abs(lhs - rhs) < 1e-6 * scale, (trial, lhs, rhs, scale)  # measured 3e-8: fp32 constants in the blob, O(eps^2) differences


def test_rodent_gravity_forces_are_the_gradient_of_the_potential(rodent, oracle_mod):
    """At rest the bias force is pure gravity, and by virtual work its i-th component is the derivative of V = sum_b m_b g z_b along
    dof i (free joint: world translation / body-frame rotation; hinges: angle) -- all 73 components against central differences of
    the forward kinematics."""
    from conftest import start_states
    A = rodent["model"].arrays
    blob, dims = rodent["model_blob"], rodent["dims"]
    mass = A["body_mass"].astype(np.float64)
    qpos, _, _ = start_states(rodent, 1, seed=31)
    qpos = qpos.astype(np.float64)
    zero = np.zeros((1, 73))
    fd = lambda q: oracle_mod.forward_dump(blob, dict(qpos=q, qvel=zero, act=np.zeros((1, 30)), qacc_warmstart=zero), None, precision=64, dims=dims)
    V = lambda d: 9.81 * float(mass @ d["xipos"][0][:, 2])

    def moved(q, i, eps):
        q = q.copy()
        if i < 3:
            q[0, i] += eps
        elif i < 6:
            w = np.zeros(3); w[i - 3] = 1.0
            q[0, 3:7] = mjcf.quat_mul(q[0, 3:7], np.concatenate([[math.cos(eps / 2)], math.sin(eps / 2) * w]))
        else:
            q[0, 7 + (i - 6)] += eps
        return q

    bias = fd(qpos)["qfrc_bias"][0]
    eps = 1e-5
    grad = np.array([(V(fd(moved(qpos, i, eps))) - V(fd(moved(qpos, i, -eps)))) / (2 * eps) for i in range(73)])
    assert np.abs(bias - grad).max() < 1e-6 * np.abs(grad).max(), np.abs(bias - grad).max() / np.abs(grad).max()
    assert abs(bias[2] - 9.81 * mass.sum()) < 1e-6 * 9.81 * mass.sum() and np.abs(bias[:2]).max() < 1e-9  # the weight, on the z dof


def test_rodent_limit_rows(rodent, oracle_mod):
    """Joint-limit rows of the rodent: J = +1 on the dof at the lower stop (pos = q - lo), -1 at the upper (pos = hi - q);
    D = imp / ((1 - imp) dof_invweight0), aref = -b (J v) - k imp pos with the joint's solref / solimp."""
    from conftest import start_states
    m = rodent["model"]
    A = m.arrays
    blob, dims = rodent["model_blob"], rodent["dims"]
    rng = np.random.default_rng(2)
    qpos, qvel, _ = start_states(rodent, 1, seed=13)
    qpos = qpos.astype(np.float64); qvel = qvel.astype(np.float64)
    lim = [j for j in range(m.njnt) if A["jnt_limited"][j] and A["jnt_type"][j] != 0]
    for j in lim[::2]:  # push every other limited joint past one of its stops
        lo, hi = A["jnt_range"][j]
        qpos[0, A["jnt_qposadr"][j]] = (lo - 0.01) if rng.random() < 0.5 else (hi + 0.02)
    d = oracle_mod.forward_dump(blob, dict(qpos=qpos, qvel=qvel, act=np.zeros((1, 30)), qacc_warmstart=np.zeros((1, 73))), None,
                                precision=64, dims=dims)
    J, pos, D, aref = d["efc_J"][0], d["efc_pos"][0], d["efc_D"][0], d["efc_aref"][0]
    nl, seen = dims["nlimit"], 0
    for r in range(nl):
        if np.abs(J[r]).max() == 0:
            continue
        i = int(np.argmax(np.abs(J[r])))
        assert np.count_nonzero(J[r]) == 1 and abs(abs(J[r][i]) - 1) < 1e-12
        j = int(A["dof_jntid"][i])
        q = qpos[0, A["jnt_qposadr"][j]]
        lo, hi = A["jnt_range"][j]
        want_pos = (q - lo) if J[r][i] > 0 else (hi - q)
        assert want_pos < 0 and abs(pos[r] - want_pos) < 1e-7, (r, pos[r], want_pos)  # range stored in fp32
        k, b = _kb(A["jnt_solref"][j], A["jnt_solimp"][j], m.timestep)
        imp = _impedance(A["jnt_solimp"][j], pos[r])
        assert abs(D[r] - imp / ((1 - imp) * A["dof_invweight0"][i])) < 2e-6 * D[r]
        assert abs(aref[r] - (-b * J[r][i] * qvel[0, i] - k * imp * pos[r])) < 1e-6 * max(1.0, abs(aref[r]))
        seen += 1
    assert seen >= len(lim[::2])  # every joint pushed past a stop produced its row
