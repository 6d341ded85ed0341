"""Checks of the robot constants that do NOT go through tools/gen_robot_model.py (VERDICT r1, weak #2: the oracle and the
kernels include byte-identical generated tables, so pinocchio's joint ordering / fixed-joint merging was invisible to
every parity test).

Here the URDF itself is parsed again, with different code and different mathematics:

  * every link stays its own rigid body (NO merging across fixed joints), the joint origins are composed with the
    textbook Rz(yaw) Ry(pitch) Rx(roll) matrices (the generator goes through urdfdom's quaternion formula);
  * the dynamics are LAGRANGIAN: kinetic + potential energy of every URDF link from its world-frame Jacobians,
    tau = d/dt(dL/dqd) - dL/dq evaluated with central differences of the energy terms -- no recursive Newton-Euler,
    no spatial algebra, no composite inertias (SURVEY 8c(i) "energy / Lagrangian check");
  * joint order = depth-first traversal with the children of a link sorted by JOINT NAME, which is what
    pinocchio::urdf::buildModel sees: urdfdom keeps joints in a std::map<std::string, ...> and fills
    Link::child_joints in that (alphabetical) order.

Needs the reference's URDF files, stored as tests/golden/iiwa14.urdf (idocp's examples/iiwa14/iiwa_description/urdf/iiwa14.urdf)
and tests/golden/anymal.urdf (examples/anymal/anymal_b_simple_description/urdf/anymal.urdf); skipped (loudly) while they are
absent.  include/idocp_b200/idocp_b200.hpp holds the content hashes of both files (kUrdfHashIiwa14, kUrdfHashAnymalExamples);
tests/test_cpp_host.py checks a stored iiwa14.urdf against its hash."""
import math
import os
import xml.etree.ElementTree as ET

import numpy as np
import pytest

from conftest import GOLDEN

IIWA_URDF = os.path.join(GOLDEN, "iiwa14.urdf")
ANYMAL_URDF = os.path.join(GOLDEN, "anymal.urdf")
G = 9.81

pytestmark = pytest.mark.skipif(not (os.path.exists(IIWA_URDF) and os.path.exists(ANYMAL_URDF)),
                                reason="tests/golden/iiwa14.urdf and anymal.urdf (idocp's URDF files) not present: "
                                       "independent model check NOT run")


def _floats(s, n):
    v = [float(x) for x in s.split()]
    assert len(v) == n
    return np.array(v)


def _rpy(r, p, y):
    cr, sr, cp, sp, cy, sy = math.cos(r), math.sin(r), math.cos(p), math.sin(p), math.cos(y), math.sin(y)
    Rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
    Ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
    Rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]])
    return Rz @ Ry @ Rx


def _origin(elem):
    o = elem.find("origin") if elem is not None else None
    if o is None:
        return np.eye(3), np.zeros(3)
    return _rpy(*_floats(o.get("rpy", "0 0 0"), 3)), _floats(o.get("xyz", "0 0 0"), 3)


class UrdfTree:
    """All links of the URDF as separate bodies; movable joints numbered by the name-sorted depth-first traversal."""

    def __init__(self, path, floating_base):
        root = ET.parse(path).getroot()
        self.links = {}
        for L in root.findall("link"):
            inertial = L.find("inertial")
            if inertial is None:
                self.links[L.get("name")] = None
                continue
            R, p = _origin(inertial)
            I = inertial.find("inertia")
            Ic = np.array([[float(I.get("ixx")), float(I.get("ixy")), float(I.get("ixz"))],
                           [float(I.get("ixy")), float(I.get("iyy")), float(I.get("iyz"))],
                           [float(I.get("ixz")), float(I.get("iyz")), float(I.get("izz"))]])
            self.links[L.get("name")] = (float(inertial.find("mass").get("value")), R, p, Ic)
        self.joints = {}
        children = set()
        for J in root.findall("joint"):
            R, p = _origin(J)
            axis = _floats(J.find("axis").get("xyz"), 3) if J.find("axis") is not None else np.array([1.0, 0, 0])
            self.joints[J.get("name")] = dict(type=J.get("type"), parent=J.find("parent").get("link"),
                                              child=J.find("child").get("link"), R=R, p=p, axis=axis)
            children.add(J.find("child").get("link"))
        roots = [n for n in self.links if n not in children]
        assert len(roots) == 1
        self.root = roots[0]
        self.floating = floating_base
        self.movable = []          # names of the revolute joints in model order
        self.order = []            # (joint name or None, link name) in traversal order
        self._walk(self.root)

    def _walk(self, link):
        for name in sorted(n for n, j in self.joints.items() if j["parent"] == link):
            j = self.joints[name]
            if j["type"] in ("revolute", "continuous"):
                self.movable.append(name)
            elif j["type"] == "floating":
                # URDF `floating` joint -> pinocchio JointModelFreeFlyer: its child link is the moving base
                assert self.floating and link == self.root and np.allclose(j["R"], np.eye(3)) and np.allclose(j["p"], 0)
                self.base = j["child"]
            else:
                assert j["type"] == "fixed", j["type"]
            self.order.append((name, j["child"]))
            self._walk(j["child"])

    # ---- kinematics of every link: world placement (R, p) as a function of the configuration ----
    def placements(self, base_R, base_p, qj):
        out = {self.root: (np.eye(3), np.zeros(3)) if self.floating else (base_R, base_p)}
        for name, child in self.order:
            j = self.joints[name]
            Rp, pp = out[j["parent"]]
            R, p = Rp @ j["R"], pp + Rp @ j["p"]
            if j["type"] == "floating":
                R, p = base_R, base_p
            if name in self.movable:
                th = qj[self.movable.index(name)]
                a = j["axis"] / np.linalg.norm(j["axis"])
                K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
                R = R @ (np.eye(3) + math.sin(th) * K + (1 - math.cos(th)) * (K @ K))      # Rodrigues
            out[child] = (R, p)
        return out

    def bodies(self, base_R, base_p, qj):
        """[(mass, world com, world inertia about the com, world rotation of the link)] of the links with mass."""
        pl = self.placements(base_R, base_p, qj)
        out = []
        for name, inertial in self.links.items():
            if inertial is None:
                continue
            m, Ri, pi, Ic = inertial
            R, p = pl[name]
            Rw = R @ Ri
            out.append((m, p + R @ pi, Rw @ Ic @ Rw.T, R))
        return out


def _skew(w):
    return np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])


def _expm_so3(w):
    th = np.linalg.norm(w)
    if th < 1e-14:
        return np.eye(3) + _skew(w)
    K = _skew(w / th)
    return np.eye(3) + math.sin(th) * K + (1 - math.cos(th)) * (K @ K)


def _quat_to_R(x, y, z, w):
    n = math.sqrt(x * x + y * y + z * z + w * w)
    x, y, z, w = x / n, y / n, z / n, w / n
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


class Lagrangian:
    """tau = M(c) a + [d/dt M] v - dT/dc + dV/dc on the configuration manifold, all derivatives by central differences of
    the energies / the mass matrix.  Coordinates: fixed base c = joint angles; floating base c = (base placement, joint
    angles) perturbed by LOCAL twists [linear; angular] in the base frame = pinocchio's free-flyer tangent space."""

    def __init__(self, tree):
        self.t = tree
        self.nv = len(tree.movable) + (6 if tree.floating else 0)

    def _split(self, c):
        if self.t.floating:
            return c[0], c[1], c[2]
        return np.eye(3), np.zeros(3), c

    def move(self, c, dv):
        """configuration reached from c along the tangent vector dv (exponential of the base twist, joint angles add)."""
        if not self.t.floating:
            return c + dv
        R, p, qj = c
        w, v = dv[3:6], dv[0:3]
        th = np.linalg.norm(w)
        if th < 1e-12:
            V = np.eye(3) + 0.5 * _skew(w)
        else:
            K = _skew(w)
            V = np.eye(3) + (1 - math.cos(th)) / th ** 2 * K + (th - math.sin(th)) / th ** 3 * (K @ K)
        return (R @ _expm_so3(w), p + R @ (V @ v), qj + dv[6:])

    def potential(self, c):
        R, p, qj = self._split(c)
        return sum(m * G * com[2] for m, com, _, _ in self.t.bodies(R, p, qj))

    def mass_matrix(self, c, h=1e-6):
        """M = sum_bodies m Jc^T Jc + Jw^T I Jw with the Jacobians from central differences of the link placements."""
        R, p, qj = self._split(c)
        nb = len(self.t.bodies(R, p, qj))
        Jc = np.zeros((nb, 3, self.nv))
        Jw = np.zeros((nb, 3, self.nv))
        base = self.t.bodies(R, p, qj)
        for k in range(self.nv):
            e = np.zeros(self.nv)
            e[k] = h
            bp = self.t.bodies(*self._split(self.move(c, e)))
            bm = self.t.bodies(*self._split(self.move(c, -e)))
            for i in range(nb):
                Jc[i, :, k] = (bp[i][1] - bm[i][1]) / (2 * h)
                dR = (bp[i][3] - bm[i][3]) / (2 * h) @ base[i][3].T           # [w]x in the world frame
                Jw[i, :, k] = [dR[2, 1], dR[0, 2], dR[1, 0]]
        M = np.zeros((self.nv, self.nv))
        for i, (m, _, Iw, _) in enumerate(base):
            M += m * Jc[i].T @ Jc[i] + Jw[i].T @ Iw @ Jw[i]
        return M

    def kinetic(self, c, v):
        return 0.5 * v @ self.mass_matrix(c) @ v

    def tau(self, c, v, a, h=1e-4):
        # Euler-Lagrange in quasi-velocities (Hamel / Euler-Poincare): d/dt(dT/dv) - ad*_v (dT/dv) - dT/dc + dV/dc
        M = self.mass_matrix(c)
        Mdot = (self.mass_matrix(self.move(c, h * v)) - self.mass_matrix(self.move(c, -h * v))) / (2 * h)
        mom = M @ v
        dT = np.zeros(self.nv)
        dV = np.zeros(self.nv)
        for k in range(self.nv):
            e = np.zeros(self.nv)
            e[k] = h
            cp, cm = self.move(c, e), self.move(c, -e)
            dT[k] = (self.kinetic(cp, v) - self.kinetic(cm, v)) / (2 * h)
            dV[k] = (self.potential(cp) - self.potential(cm)) / (2 * h)
        tau = M @ a + Mdot @ v - dT + dV
        if self.t.floating:
            # coadjoint term of the base twist (v = [lin; ang] in the base frame): -ad*_v (dT/dv)
            vl, vw, pl, pw = v[0:3], v[3:6], mom[0:3], mom[3:6]
            tau[0:3] += np.cross(vw, pl)
            tau[3:6] += np.cross(vw, pw) + np.cross(vl, pl)
        return tau


def test_iiwa14_joint_order_and_lagrangian_torques(oracle):
    tree = UrdfTree(IIWA_URDF, floating_base=False)
    assert tree.movable == ["iiwa_joint_%d" % i for i in range(1, 8)]
    lag = Lagrangian(tree)
    rng = np.random.default_rng(5)
    for _ in range(3):
        q, v, a = rng.uniform(-2, 2, 7), rng.uniform(-2, 2, 7), rng.uniform(-4, 4, 7)
        tau = lag.tau(q, v, a)
        ref = oracle.rnea(q, v, a)
        assert np.max(np.abs(tau - ref)) < 2e-5 * max(1.0, np.max(np.abs(ref))), (tau, ref)
    # total mass of every URDF link (merged or not) and the mass matrix against dtau/da of the oracle
    assert abs(sum(x[0] for x in tree.links.values() if x) - 5.0 - sum([4, 4, 3, 2.7, 1.7, 1.8, 0.3])) < 1e-12
    q = rng.uniform(-2, 2, 7)
    _, _, Mo = oracle.rnea_derivatives(q, np.zeros(7), np.zeros(7))
    assert np.max(np.abs(lag.mass_matrix(q) - Mo)) < 1e-7


def test_anymal_joint_order_and_lagrangian_torques(oracle):
    import fb_py
    fb_py.lib()
    tree = UrdfTree(ANYMAL_URDF, floating_base=True)
    assert tree.movable == [leg + "_" + j for leg in ("LF", "LH", "RF", "RH") for j in ("HAA", "HFE", "KFE")]
    lag = Lagrangian(tree)
    rng = np.random.default_rng(6)
    total = sum(x[0] for x in tree.links.values() if x)
    import anymal_problems
    assert abs(total * G - anymal_problems.TOTAL_WEIGHT) < 1e-9      # Robot::totalWeight used by the examples' f_ref
    for _ in range(2):
        quat = rng.normal(size=4)
        quat /= np.linalg.norm(quat)
        p, qj = rng.uniform(-1, 1, 3), rng.uniform(-1, 1, 12)
        v, a = rng.uniform(-1, 1, 18), rng.uniform(-2, 2, 18)
        q = np.concatenate([p, quat, qj])
        ref = fb_py.rnea(q, v, a)
        tau = lag.tau((_quat_to_R(*quat), p, qj), v, a)
        assert np.max(np.abs(tau - ref)) < 5e-5 * max(1.0, np.max(np.abs(ref))), (tau - ref)
    quat = np.array([0, 0, 0, 1.0])
    q = np.concatenate([np.zeros(3), quat, np.zeros(12)])
    _, _, _, Mo = fb_py.rnea(q, np.zeros(18), np.zeros(18), derivatives=True)
    assert np.max(np.abs(lag.mass_matrix((np.eye(3), np.zeros(3), np.zeros(12))) - Mo)) < 1e-6


def test_contact_frames_from_the_urdf(oracle):
    """The feet: position of LF/LH/RF/RH_FOOT in the world from the raw URDF chain vs the oracle's contact kinematics."""
    import fb_py
    fb_py.lib()
    tree = UrdfTree(ANYMAL_URDF, floating_base=True)
    rng = np.random.default_rng(8)
    quat = rng.normal(size=4)
    quat /= np.linalg.norm(quat)
    p, qj = rng.uniform(-1, 1, 3), rng.uniform(-1, 1, 12)
    pl = tree.placements(_quat_to_R(*quat), p, qj)
    q = np.concatenate([p, quat, qj])
    z = np.zeros(18)
    for i, foot in enumerate(("LF_FOOT", "LH_FOOT", "RF_FOOT", "RH_FOOT")):
        P = fb_py.contact(q, z, z, i, 0.05, np.zeros(3))["P"]
        assert np.allclose(P, pl[foot][1], rtol=0, atol=1e-12), foot
