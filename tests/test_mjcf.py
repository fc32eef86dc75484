"""CPU suite: the MJCF importer (abr_control_b200/arms/mjcf.py, SURVEY.md S8f row 4).

MuJoCo is not in this image, so the importer cannot be compared with ``MujocoConfig`` itself (SURVEY.md S8c: that path is
"parity unpinned").  It is checked (i) by a round trip: a random serial chain is written out as MJCF (body pos/quat,
joint pos/axis, inertial pos/quat/mass/diaginertia, an EE body) and read back — the oracle built from the imported
descriptor must reproduce, for random joint angles, the world poses computed directly from the numbers that went into
the file; (ii) on the reference's own UR5 model (tests/golden/ur5_mjcf.xml: its ``ur5.xml`` without geometry): the zero
pose is the sum of the body offsets in the file, and each joint moves the end effector about the axis the file names.
"""
import os

import numpy as np
import pytest

from abr_control_b200.arms.mjcf import chain_desc_from_mjcf
from oracle import rbd_oracle as ro


def _rot(axis, ang):
    a = np.asarray(axis, dtype=float) / np.linalg.norm(axis)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(ang) * K + (1 - np.cos(ang)) * K @ K


def _quat(R):
    w = np.sqrt(max(0.0, 1 + R[0, 0] + R[1, 1] + R[2, 2])) / 2
    if w > 1e-6:
        return np.array([w, (R[2, 1] - R[1, 2]) / (4 * w), (R[0, 2] - R[2, 0]) / (4 * w), (R[1, 0] - R[0, 1]) / (4 * w)])
    vals, vecs = np.linalg.eigh((R + R.T) / 2)
    ax = vecs[:, -1]
    return np.array([0.0, ax[0], ax[1], ax[2]])


def _random_model(n, seed):
    rng = np.random.default_rng(seed)

    def rnd_R():
        return _rot(rng.normal(size=3), rng.uniform(0, np.pi))

    bodies = []
    for i in range(n):
        bodies.append(dict(pos=rng.uniform(-0.3, 0.3, 3), R=rnd_R(), jpos=rng.uniform(-0.05, 0.05, 3),
                           axis=rng.normal(size=3), ipos=rng.uniform(-0.1, 0.1, 3), iR=rnd_R(),
                           mass=rng.uniform(0.3, 4), di=rng.uniform(0.01, 0.2, 3)))
    ee = dict(pos=rng.uniform(-0.1, 0.1, 3), R=rnd_R())
    return bodies, ee


def _write(path, bodies, ee):
    f = lambda v: " ".join(f"{x:.17g}" for x in v)  # noqa: E731
    out = ['<mujoco model="rand"><compiler angle="radian"/>',
           '<custom><numeric name="START_ANGLES" data="%s"/></custom><worldbody><body name="base_link" pos="0.1 -0.2 0.3">'
           % " ".join("0.1" for _ in bodies)]
    for i, b in enumerate(bodies):
        out.append(f'<body name="link{i + 1}" pos="{f(b["pos"])}" quat="{f(_quat(b["R"]))}">')
        out.append(f'<joint name="joint{i}" axis="{f(b["axis"])}" pos="{f(b["jpos"])}"/>')
        out.append(f'<inertial pos="{f(b["ipos"])}" quat="{f(_quat(b["iR"]))}" mass="{b["mass"]:.17g}" diaginertia="{f(b["di"])}"/>')
    out.append(f'<body name="EE" pos="{f(ee["pos"])}" quat="{f(_quat(ee["R"]))}"/>')
    out.append("</body>" * len(bodies) + "</body></worldbody><actuator>")
    out += [f'<motor name="m{i}" joint="joint{i}"/>' for i in range(len(bodies))]
    out.append("</actuator></mujoco>")
    open(path, "w").write("\n".join(out))


def _direct_fk(bodies, ee, q):
    """world poses from the model's own numbers: body i = parent . T(pos, R) . [rotation by q_i about axis through jpos]"""
    T = np.eye(4)
    T[:3, 3] = [0.1, -0.2, 0.3]
    coms, joints = [], []
    for b, qi in zip(bodies, q):
        Tb = np.eye(4)
        Tb[:3, :3], Tb[:3, 3] = b["R"], b["pos"]
        T = T @ Tb
        joints.append((T @ np.append(b["jpos"], 1))[:3])
        Rq = np.eye(4)
        Rq[:3, :3] = _rot(b["axis"], qi)
        Rq[:3, 3] = b["jpos"] - Rq[:3, :3] @ b["jpos"]
        T = T @ Rq
        coms.append((T @ np.append(b["ipos"], 1))[:3])
    Te = np.eye(4)
    Te[:3, :3], Te[:3, 3] = ee["R"], ee["pos"]
    return coms, joints, T @ Te


@pytest.mark.parametrize("n", [2, 4, 6, 7])
def test_round_trip_through_an_mjcf_file(tmp_path, n):
    bodies, ee = _random_model(n, 10 + n)
    path = str(tmp_path / "rand.xml")
    _write(path, bodies, ee)
    desc = chain_desc_from_mjcf(path)
    assert desc["n_joints"] == n and desc["n_links"] == n + 1 and desc["start_angles"] == [0.1] * n
    c = ro.ChainOracle(desc)
    rng = np.random.default_rng(n)
    for q in rng.uniform(-np.pi, np.pi, (6, n)):
        coms, joints, Tee = _direct_fk(bodies, ee, q)
        assert np.abs(c.Tx("EE", q[None])[0] - Tee[:3, 3]).max() < 1e-12
        assert np.abs(c.R("EE", q[None])[0] - Tee[:3, :3]).max() < 1e-12
        for i in range(n):
            assert np.abs(c.Tx(f"link{i + 1}", q[None])[0] - coms[i]).max() < 1e-12
            assert np.abs(c.Tx(f"joint{i}", q[None])[0] - joints[i]).max() < 1e-12
    li = np.array(desc["link_inertia"])
    assert np.allclose(li[1:, 0], [b["mass"] for b in bodies]) and np.allclose(li[1:, 3:], [b["di"] for b in bodies])


UR5_XML = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ur5_mjcf.xml")


def test_reference_ur5_xml():
    desc = chain_desc_from_mjcf(UR5_XML)
    assert desc["n_joints"] == 6 and desc["joint_names"] == [f"joint{i}" for i in range(6)]
    assert desc["start_angles"] == [0.0, -0.67, -0.67, 0.0, 0.0, 0.0]
    c = ro.ChainOracle(desc)
    offsets = np.array([[0, 0, 0.0213], [-0.0663, 0, 0.0679], [-0.008, 0, 0.425], [0.0173, 0, 0.3922],
                        [-0.05325, 0, 0.04165], [-0.04165, 0, 0.05305], [-0.04, 0, 0]])
    assert np.abs(c.Tx("EE", np.zeros((1, 6)))[0] - offsets.sum(axis=0)).max() < 1e-12  # the file's own numbers
    axes = [[0, 0, 1], [-1, 0, 0], [1, 0, 0], [-1, 0, 0], [0, 0, 1], [-1, 0, 0]]  # every body frame is world aligned at zero
    J = c.J("EE", np.zeros((1, 6)))[0]
    assert np.abs(J[3:].T - np.array(axes, dtype=float)).max() < 1e-12
    masses = [3.761, 8.058, 2.846, 1.37, 1.3, 0.365]
    assert np.allclose(np.array(desc["link_inertia"])[1:, 0], masses)
