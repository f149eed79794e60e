"""MJCF subset front-end: FARMS-schema MJCF text -> flat ``Model``.

The reference hands its MJCF tree to ``dm_control.mjcf.Physics.from_mjcf_model``
(farms_mujoco/simulation/simulation.py:53), i.e. to the MuJoCo compiler (third
party, absent here).  This module ingests the *schema the reference's builder
emits* (farms_mujoco/simulation/mjcf.py:132-600, 647-1035, 1245-1481; SURVEY.md
section 3.5) and performs the compiler steps that change numbers (SURVEY.md
Appendix A.9): principal-axis inertias, qpos0/qpos_spring, dof tree, sparse
mass-matrix addresses, dof_invweight0/body_invweight0, geom_rbound, static-body
fusing, plane-vs-primitive collision candidates with mixed contact parameters.

Supported: one kinematic tree (free or fixed base), <=1 joint per body
(free/hinge/slide), sphere/capsule collision geoms against world planes,
position/velocity/motor actuators with joint transmission, the sensor types the
reference reads (framelinvel/frameangvel/framepos/framequat with objtype=body,
jointpos/jointvel/jointlimitfrc, actuatorfrc), one keyframe.
Everything else the builder can emit (meshes, hfields, tendons/muscles,
cameras, lights, textures) is init-time or rendering and is ignored or rejected
with an explicit error.
"""

import copy
import xml.etree.ElementTree as ET
from dataclasses import dataclass, field
from typing import Dict, List

import numpy as np

# MuJoCo enums (mjtJoint, mjtGeom) kept so logs/maps read like the reference's
JNT_FREE, JNT_BALL, JNT_SLIDE, JNT_HINGE = 0, 1, 2, 3
GEOM_PLANE, GEOM_HFIELD, GEOM_SPHERE, GEOM_CAPSULE = 0, 1, 2, 3
GEOM_ELLIPSOID, GEOM_CYLINDER, GEOM_BOX, GEOM_MESH = 4, 5, 6, 7
GEOM_TYPES = {
    'plane': GEOM_PLANE, 'hfield': GEOM_HFIELD, 'sphere': GEOM_SPHERE,
    'capsule': GEOM_CAPSULE, 'ellipsoid': GEOM_ELLIPSOID,
    'cylinder': GEOM_CYLINDER, 'box': GEOM_BOX, 'mesh': GEOM_MESH,
}
ACT_POSITION, ACT_VELOCITY, ACT_MOTOR = 0, 1, 2
SENS_FRAMEPOS, SENS_FRAMEQUAT, SENS_FRAMELINVEL, SENS_FRAMEANGVEL = 0, 1, 2, 3
SENS_JOINTPOS, SENS_JOINTVEL, SENS_JOINTLIMITFRC, SENS_ACTUATORFRC = 4, 5, 6, 7
SENSOR_TYPES = {
    'framepos': (SENS_FRAMEPOS, 3), 'framequat': (SENS_FRAMEQUAT, 4),
    'framelinvel': (SENS_FRAMELINVEL, 3), 'frameangvel': (SENS_FRAMEANGVEL, 3),
    'jointpos': (SENS_JOINTPOS, 1), 'jointvel': (SENS_JOINTVEL, 1),
    'jointlimitfrc': (SENS_JOINTLIMITFRC, 1),
    'actuatorfrc': (SENS_ACTUATORFRC, 1),
}

# MuJoCo constants (third party; isolated here and in csrc/fb_constants.h)
MJ_MINVAL = 1e-15
MJ_MINMU = 1e-5
DEFAULT_SOLREF = (0.02, 1.0)
DEFAULT_SOLIMP = (0.9, 0.95, 0.001, 0.5, 2.0)


# --------------------------------------------------------------------------
# Small quaternion / rotation helpers (MuJoCo convention: w, x, y, z)
# --------------------------------------------------------------------------

def quat_mul(a, b):
    """Hamilton product, wxyz."""
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return np.array([
        aw*bw - ax*bx - ay*by - az*bz,
        aw*bx + ax*bw + ay*bz - az*by,
        aw*by - ax*bz + ay*bw + az*bx,
        aw*bz + ax*by - ay*bx + az*bw,
    ])


def quat2mat(q):
    """Rotation matrix of a unit quaternion, wxyz."""
    w, x, y, z = q
    return np.array([
        [w*w + x*x - y*y - z*z, 2*(x*y - w*z), 2*(x*z + w*y)],
        [2*(x*y + w*z), w*w - x*x + y*y - z*z, 2*(y*z - w*x)],
        [2*(x*z - w*y), 2*(y*z + w*x), w*w - x*x - y*y + z*z],
    ])


def mat2quat(mat):
    """Unit quaternion (wxyz) of a proper rotation matrix."""
    m = np.asarray(mat, dtype=float)
    tr = m[0, 0] + m[1, 1] + m[2, 2]
    if tr > 0:
        s = np.sqrt(tr + 1.0)*2
        q = [0.25*s, (m[2, 1] - m[1, 2])/s, (m[0, 2] - m[2, 0])/s, (m[1, 0] - m[0, 1])/s]
    elif m[0, 0] > m[1, 1] and m[0, 0] > m[2, 2]:
        s = np.sqrt(1.0 + m[0, 0] - m[1, 1] - m[2, 2])*2
        q = [(m[2, 1] - m[1, 2])/s, 0.25*s, (m[0, 1] + m[1, 0])/s, (m[0, 2] + m[2, 0])/s]
    elif m[1, 1] > m[2, 2]:
        s = np.sqrt(1.0 + m[1, 1] - m[0, 0] - m[2, 2])*2
        q = [(m[0, 2] - m[2, 0])/s, (m[0, 1] + m[1, 0])/s, 0.25*s, (m[1, 2] + m[2, 1])/s]
    else:
        s = np.sqrt(1.0 + m[2, 2] - m[0, 0] - m[1, 1])*2
        q = [(m[1, 0] - m[0, 1])/s, (m[0, 2] + m[2, 0])/s, (m[1, 2] + m[2, 1])/s, 0.25*s]
    q = np.array(q)
    return q/np.linalg.norm(q)


def axisangle2quat(axis, angle):
    axis = np.asarray(axis, dtype=float)
    return np.concatenate([[np.cos(0.5*angle)], np.sin(0.5*angle)*axis])


def euler_xyz2quat(euler):
    """Intrinsic-free 'xyz' Euler (scipy lower-case = extrinsic) -> wxyz.

    Mirrors ``euler2mjcquat`` of the reference (mjcf.py:47-52), which uses
    ``Rotation.from_euler(seq='xyz')``: R = Rz(c) @ Ry(b) @ Rx(a).
    """
    a, b, c = euler
    qx = axisangle2quat([1, 0, 0], a)
    qy = axisangle2quat([0, 1, 0], b)
    qz = axisangle2quat([0, 0, 1], c)
    return quat_mul(qz, quat_mul(qy, qx))


def _floats(text, n=None, default=None):
    if text is None:
        return None if default is None else np.array(default, dtype=float)
    vals = np.array([float(v) for v in text.replace(',', ' ').split()], dtype=float)
    if n is not None and len(vals) != n:
        raise ValueError(f'expected {n} numbers, got "{text}"')
    return vals


def _bool(text, default=False):
    if text is None:
        return default
    return text.strip().lower() in ('true', '1')


# --------------------------------------------------------------------------
# Flat model
# --------------------------------------------------------------------------

@dataclass
class Model:
    """Flat, compiled model (the ``mjModel`` subset the hot path reads)."""
    # pylint: disable=too-many-instance-attributes
    name: str = ''
    # options
    timestep: float = 0.002
    gravity: np.ndarray = None
    impratio: float = 1.0
    cone: str = 'pyramidal'
    solver: str = 'Newton'
    iterations: int = 100
    tolerance: float = 1e-8
    integrator: str = 'Euler'
    # bodies
    body_names: List[str] = field(default_factory=list)
    body_parentid: np.ndarray = None
    body_pos: np.ndarray = None
    body_quat: np.ndarray = None
    body_ipos: np.ndarray = None
    body_iquat: np.ndarray = None
    body_mass: np.ndarray = None
    body_inertia: np.ndarray = None
    body_jntid: np.ndarray = None      # joint of the body or -1 (<=1 joint/body)
    body_dofadr: np.ndarray = None
    body_dofnum: np.ndarray = None
    body_depth: np.ndarray = None
    body_invweight0: np.ndarray = None
    # joints
    jnt_names: List[str] = field(default_factory=list)
    jnt_type: np.ndarray = None
    jnt_bodyid: np.ndarray = None
    jnt_qposadr: np.ndarray = None
    jnt_dofadr: np.ndarray = None
    jnt_pos: np.ndarray = None
    jnt_axis: np.ndarray = None
    jnt_stiffness: np.ndarray = None
    jnt_limited: np.ndarray = None
    jnt_range: np.ndarray = None
    jnt_margin: np.ndarray = None
    jnt_solref: np.ndarray = None
    jnt_solimp: np.ndarray = None
    # dofs
    dof_bodyid: np.ndarray = None
    dof_jntid: np.ndarray = None
    dof_parentid: np.ndarray = None
    dof_damping: np.ndarray = None
    dof_armature: np.ndarray = None
    dof_invweight0: np.ndarray = None
    dof_Madr: np.ndarray = None
    nM: int = 0
    qpos0: np.ndarray = None
    qpos_spring: np.ndarray = None
    # geoms (collision geoms only: contype|conaffinity != 0)
    geom_names: List[str] = field(default_factory=list)
    geom_type: np.ndarray = None
    geom_bodyid: np.ndarray = None
    geom_pos: np.ndarray = None
    geom_quat: np.ndarray = None
    geom_size: np.ndarray = None
    geom_friction: np.ndarray = None
    geom_solref: np.ndarray = None
    geom_solimp: np.ndarray = None
    geom_solmix: np.ndarray = None
    geom_margin: np.ndarray = None
    geom_gap: np.ndarray = None
    geom_contype: np.ndarray = None
    geom_conaffinity: np.ndarray = None
    geom_condim: np.ndarray = None
    geom_priority: np.ndarray = None
    geom_rbound: np.ndarray = None
    # actuators
    actuator_names: List[str] = field(default_factory=list)
    actuator_kind: np.ndarray = None       # ACT_POSITION / ACT_VELOCITY / ACT_MOTOR
    actuator_trnid: np.ndarray = None      # joint id
    actuator_trntype: np.ndarray = None    # 0 = joint
    actuator_gainprm: np.ndarray = None    # [nu, 3]
    actuator_biasprm: np.ndarray = None    # [nu, 3]
    actuator_ctrllimited: np.ndarray = None
    actuator_ctrlrange: np.ndarray = None
    actuator_forcelimited: np.ndarray = None
    actuator_forcerange: np.ndarray = None
    actuator_gear: np.ndarray = None
    # sensors
    sensor_names: List[str] = field(default_factory=list)
    sensor_type: np.ndarray = None
    sensor_objid: np.ndarray = None
    sensor_adr: np.ndarray = None
    sensor_dim: np.ndarray = None
    nsensordata: int = 0
    # keyframe
    key_qpos: np.ndarray = None
    key_qvel: np.ndarray = None
    key_ctrl: np.ndarray = None
    # collision candidates (plane vs sphere / capsule end), compile-time
    cand_geom1: np.ndarray = None      # plane geom id
    cand_geom2: np.ndarray = None      # animat geom id
    cand_end: np.ndarray = None        # 0 sphere centre, +1 / -1 capsule ends, 2..9 box corner (end - 2), 10 ellipsoid, 11..14 cylinder points,
                                       # 20 sphere-sphere <pair>, 21 frictionless sphere-sphere <pair> solved as a hard normal row
    cand_friction: np.ndarray = None   # mixed sliding friction
    cand_solref: np.ndarray = None     # [ncand, 2]
    cand_solimp: np.ndarray = None     # [ncand, 5]
    cand_margin: np.ndarray = None     # mixed margin
    cand_gap: np.ndarray = None
    # statistics
    meaninertia: float = 1.0

    @property
    def nbody(self):
        return len(self.body_names)

    @property
    def njnt(self):
        return len(self.jnt_names)

    @property
    def nq(self):
        return len(self.qpos0)

    @property
    def nv(self):
        return len(self.dof_bodyid)

    @property
    def nu(self):
        return len(self.actuator_names)

    @property
    def ngeom(self):
        return len(self.geom_names)

    @property
    def ncand(self):
        return len(self.cand_geom2)

    # named lookups (dm_control ``physics.named...axes.row`` stand-ins) -----
    def body_id(self, name):
        return self.body_names.index(name)

    def jnt_id(self, name):
        return self.jnt_names.index(name)

    def geom_id(self, name):
        return self.geom_names.index(name)

    def actuator_id(self, name):
        return self.actuator_names.index(name)

    def sensor_id(self, name):
        return self.sensor_names.index(name)

    def qpos_names(self):
        """Row names of qpos/qvel (one per joint, as dm_control reports them)."""
        return list(self.jnt_names)


# --------------------------------------------------------------------------
# Parsing
# --------------------------------------------------------------------------

class _RawBody:
    def __init__(self, name, parent, pos, quat):
        self.name = name
        self.parent = parent
        self.pos = pos
        self.quat = quat
        self.joint = None
        self.inertial = None
        self.geoms = []
        self.children = []


def _parse_body(elem, parent, bodies, anon):
    name = elem.get('name')
    if name is None:
        name = f'_anon_body_{anon[0]}'
        anon[0] += 1
    pos = _floats(elem.get('pos'), 3, [0, 0, 0])
    if elem.get('euler') is not None:
        quat = euler_xyz2quat(_floats(elem.get('euler'), 3))
    else:
        quat = _floats(elem.get('quat'), 4, [1, 0, 0, 0])
    quat = quat/np.linalg.norm(quat)
    body = _RawBody(name, parent, pos, quat)
    bodies.append(body)
    if parent is not None:
        parent.children.append(body)
    joints = [c for c in elem if c.tag in ('joint', 'freejoint')]
    if len(joints) > 1:
        raise NotImplementedError(
            f'body "{name}": more than one joint per body is outside the '
            'FARMS schema (mjcf.py:180-212 emits one joint per link)')
    if joints:
        body.joint = joints[0]
    inertials = elem.findall('inertial')
    if inertials:
        body.inertial = inertials[0]
    body.geoms = elem.findall('geom')
    for child in elem.findall('body'):
        _parse_body(child, body, bodies, anon)
    return body


FRICTIONLESS_PAIRS = ('refuse', 'hard')


def parse_mjcf(xml_text: str, frictionless_pairs: str = 'refuse') -> Model:
    """Parse FARMS-schema MJCF text and compile it into a flat ``Model``.

    ``frictionless_pairs`` says what becomes of a ``<contact><pair>`` whose friction is at MuJoCo's
    floor (``friction="0 ..."``, what the reference writes for every self-collision):
    ``'refuse'`` (default) raises, ``'hard'`` compiles it to a hard normal row (candidate kind 21)
    that drops the O(mu) terms of the pyramidal cone (DESIGN.md section 8)."""
    # pylint: disable=too-many-locals,too-many-branches,too-many-statements
    if frictionless_pairs not in FRICTIONLESS_PAIRS:
        raise ValueError(f'frictionless_pairs must be one of {FRICTIONLESS_PAIRS}, not {frictionless_pairs!r}')
    root = ET.fromstring(xml_text)
    if root.tag != 'mujoco':
        raise ValueError('not an MJCF document')
    if root.find('default') is not None and len(root.find('default')):
        raise NotImplementedError('<default> classes are not part of the FARMS schema')
    compiler = root.find('compiler')
    if compiler is not None:
        if compiler.get('angle', 'radian') != 'radian':
            raise NotImplementedError('compiler angle must be radian (mjcf.py:1246)')
        if _bool(compiler.get('inertiafromgeom'), False):
            raise NotImplementedError('inertiafromgeom must be false (mjcf.py:1251)')
    fusestatic = True if compiler is None else _bool(compiler.get('fusestatic'), True)

    model = Model(name=root.get('model', ''))
    model.gravity = np.array([0, 0, -9.81])
    option = root.find('option')
    if option is not None:
        model.timestep = float(option.get('timestep', model.timestep))
        model.gravity = _floats(option.get('gravity'), 3, model.gravity)
        model.impratio = float(option.get('impratio', 1.0))
        model.cone = option.get('cone', 'pyramidal')
        model.solver = option.get('solver', 'Newton')
        model.iterations = int(option.get('iterations', 100))
        model.tolerance = float(option.get('tolerance', 1e-8))
        model.integrator = option.get('integrator', 'Euler')
    if model.cone != 'pyramidal':
        raise NotImplementedError('only cone=pyramidal (the builder fallback, mjcf.py:1342-1347)')
    if model.integrator != 'Euler':
        raise NotImplementedError('only integrator=Euler (the builder fallback, mjcf.py:1360-1365)')

    # ---- bodies ----------------------------------------------------------
    worldbody = root.find('worldbody')
    raw = []
    anon = [0]
    world = _RawBody('world', None, np.zeros(3), np.array([1., 0, 0, 0]))
    raw.append(world)
    world.geoms = worldbody.findall('geom')
    for child in worldbody.findall('body'):
        _parse_body(child, world, raw, anon)

    # names referenced by sensors keep their body (fusestatic is disabled for
    # referenced bodies in MuJoCo)
    sensor_root = root.find('sensor')
    referenced = set()
    if sensor_root is not None:
        for sens in sensor_root:
            if sens.get('objtype', 'body') == 'body' and sens.get('objname'):
                referenced.add(sens.get('objname'))

    # static = no joint anywhere between the body and the world
    def is_static(body):
        while body is not None and body is not world:
            if body.joint is not None:
                return False
            body = body.parent
        return True

    kept = [world]
    world_geoms = [(g, np.zeros(3), np.array([1., 0, 0, 0])) for g in world.geoms]
    fused_into = {}

    def world_pose(body):
        chain = []
        while body is not None and body is not world:
            chain.append(body)
            body = body.parent
        pos = np.zeros(3)
        quat = np.array([1., 0, 0, 0])
        for b in reversed(chain):
            pos = pos + quat2mat(quat) @ b.pos
            quat = quat_mul(quat, b.quat)
        return pos, quat

    for body in raw[1:]:
        if fusestatic and is_static(body) and body.name not in referenced:
            pos, quat = world_pose(body)
            for geom in body.geoms:
                world_geoms.append((geom, pos, quat))
            fused_into[body.name] = 'world'
            continue
        # re-root bodies whose ancestors were fused onto the nearest kept ancestor
        while body.parent is not world and body.parent.name in fused_into:
            par = body.parent
            body.pos = par.pos + quat2mat(par.quat) @ body.pos
            body.quat = quat_mul(par.quat, body.quat)
            body.parent = par.parent
        kept.append(body)

    index = {id(b): i for i, b in enumerate(kept)}
    nbody = len(kept)
    model.body_names = [b.name for b in kept]
    model.body_parentid = np.zeros(nbody, dtype=np.int32)
    model.body_pos = np.zeros((nbody, 3))
    model.body_quat = np.tile([1., 0, 0, 0], (nbody, 1))
    model.body_ipos = np.zeros((nbody, 3))
    model.body_iquat = np.tile([1., 0, 0, 0], (nbody, 1))
    model.body_mass = np.zeros(nbody)
    model.body_inertia = np.zeros((nbody, 3))
    model.body_jntid = -np.ones(nbody, dtype=np.int32)
    model.body_dofadr = -np.ones(nbody, dtype=np.int32)
    model.body_dofnum = np.zeros(nbody, dtype=np.int32)
    model.body_depth = np.zeros(nbody, dtype=np.int32)

    jnt = dict(names=[], type=[], bodyid=[], qposadr=[], dofadr=[], pos=[], axis=[],
               stiffness=[], limited=[], range=[], margin=[], solref=[], solimp=[],
               damping=[], armature=[], ref=[], springref=[])
    nq = 0
    nv = 0
    for i, body in enumerate(kept):
        if i == 0:
            continue
        parent = body.parent
        model.body_parentid[i] = index[id(parent)]
        if model.body_parentid[i] >= i:
            raise AssertionError('bodies must be in depth-first order')
        model.body_depth[i] = model.body_depth[model.body_parentid[i]] + 1
        model.body_pos[i] = body.pos
        model.body_quat[i] = body.quat
        if body.inertial is not None:
            ine = body.inertial
            model.body_ipos[i] = _floats(ine.get('pos'), 3, [0, 0, 0])
            model.body_mass[i] = float(ine.get('mass', 0))
            iquat = _floats(ine.get('quat'), 4, [1, 0, 0, 0])
            iquat = iquat/np.linalg.norm(iquat)
            if ine.get('fullinertia') is not None:
                fi = _floats(ine.get('fullinertia'), 6)
                full = np.array([[fi[0], fi[3], fi[4]],
                                 [fi[3], fi[1], fi[5]],
                                 [fi[4], fi[5], fi[2]]])
                evals, evecs = np.linalg.eigh(full)
                if evals.min() < -MJ_MINVAL:
                    raise ValueError(f'body {body.name}: inertia not positive')
                order = np.argsort(-evals)  # descending, like mju_eig3
                evals = evals[order]
                evecs = evecs[:, order]
                if np.linalg.det(evecs) < 0:
                    evecs[:, 2] *= -1
                model.body_inertia[i] = evals
                model.body_iquat[i] = quat_mul(iquat, mat2quat(evecs))
            else:
                model.body_inertia[i] = _floats(ine.get('diaginertia'), 3, [0, 0, 0])
                model.body_iquat[i] = iquat
        if body.joint is not None:
            j = body.joint
            jid = len(jnt['names'])
            model.body_jntid[i] = jid
            model.body_dofadr[i] = nv
            jtype = 'free' if j.tag == 'freejoint' else j.get('type', 'hinge')
            jnt['names'].append(j.get('name', f'_anon_joint_{jid}'))
            jnt['bodyid'].append(i)
            jnt['qposadr'].append(nq)
            jnt['dofadr'].append(nv)
            jnt['pos'].append(_floats(j.get('pos'), 3, [0, 0, 0]))
            axis = _floats(j.get('axis'), 3, [0, 0, 1])
            jnt['axis'].append(axis/max(np.linalg.norm(axis), MJ_MINVAL))
            jnt['stiffness'].append(float(j.get('stiffness', 0)))
            jnt['damping'].append(float(j.get('damping', 0)))
            jnt['armature'].append(float(j.get('armature', 0)))
            jnt['ref'].append(float(j.get('ref', 0)))
            jnt['springref'].append(float(j.get('springref', 0)))
            rng = _floats(j.get('range'), 2, [0, 0])
            limited = j.get('limited')
            if limited is None or limited == 'auto':
                limited = bool(rng[0] != 0 or rng[1] != 0)
            else:
                limited = _bool(limited)
            jnt['limited'].append(limited)
            jnt['range'].append(rng)
            jnt['margin'].append(float(j.get('margin', 0)))
            jnt['solref'].append(_floats(j.get('solreflimit'), 2, DEFAULT_SOLREF))
            jnt['solimp'].append(_floats(j.get('solimplimit'), 5, DEFAULT_SOLIMP))
            if jtype == 'free':
                jnt['type'].append(JNT_FREE)
                model.body_dofnum[i] = 6
                nq += 7
                nv += 6
            elif jtype in ('hinge', 'slide'):
                jnt['type'].append(JNT_HINGE if jtype == 'hinge' else JNT_SLIDE)
                model.body_dofnum[i] = 1
                nq += 1
                nv += 1
            else:
                raise NotImplementedError(f'joint type {jtype} is outside the FARMS schema')

    model.jnt_names = jnt['names']
    model.jnt_type = np.array(jnt['type'], dtype=np.int32)
    model.jnt_bodyid = np.array(jnt['bodyid'], dtype=np.int32)
    model.jnt_qposadr = np.array(jnt['qposadr'], dtype=np.int32)
    model.jnt_dofadr = np.array(jnt['dofadr'], dtype=np.int32)
    model.jnt_pos = np.array(jnt['pos'], dtype=float).reshape(-1, 3)
    model.jnt_axis = np.array(jnt['axis'], dtype=float).reshape(-1, 3)
    model.jnt_stiffness = np.array(jnt['stiffness'], dtype=float)
    model.jnt_limited = np.array(jnt['limited'], dtype=np.int32)
    model.jnt_range = np.array(jnt['range'], dtype=float).reshape(-1, 2)
    model.jnt_margin = np.array(jnt['margin'], dtype=float)
    model.jnt_solref = np.array(jnt['solref'], dtype=float).reshape(-1, 2)
    model.jnt_solimp = np.array(jnt['solimp'], dtype=float).reshape(-1, 5)

    # ---- dofs ------------------------------------------------------------
    model.dof_bodyid = np.zeros(nv, dtype=np.int32)
    model.dof_jntid = np.zeros(nv, dtype=np.int32)
    model.dof_parentid = -np.ones(nv, dtype=np.int32)
    model.dof_damping = np.zeros(nv)
    model.dof_armature = np.zeros(nv)
    model.qpos0 = np.zeros(nq)
    model.qpos_spring = np.zeros(nq)
    last_dof_of_body = -np.ones(nbody, dtype=np.int32)
    for i in range(1, nbody):
        last_dof_of_body[i] = last_dof_of_body[model.body_parentid[i]]
        jid = model.body_jntid[i]
        if jid < 0:
            continue
        adr = model.jnt_dofadr[jid]
        qadr = model.jnt_qposadr[jid]
        ndof = model.body_dofnum[i]
        for k in range(ndof):
            model.dof_bodyid[adr+k] = i
            model.dof_jntid[adr+k] = jid
            model.dof_parentid[adr+k] = last_dof_of_body[i] if k == 0 else adr+k-1
            model.dof_damping[adr+k] = jnt['damping'][jid] if ndof == 1 else 0.0
            model.dof_armature[adr+k] = jnt['armature'][jid]
        last_dof_of_body[i] = adr + ndof - 1
        if model.jnt_type[jid] == JNT_FREE:
            model.qpos0[qadr:qadr+3] = model.body_pos[i]
            model.qpos0[qadr+3:qadr+7] = model.body_quat[i]
            model.qpos_spring[qadr:qadr+7] = model.qpos0[qadr:qadr+7]
        else:
            model.qpos0[qadr] = jnt['ref'][jid]
            model.qpos_spring[qadr] = jnt['springref'][jid]
    model.dof_Madr = np.zeros(nv, dtype=np.int32)
    adr = 0
    for d in range(nv):
        model.dof_Madr[d] = adr
        k = d
        while k >= 0:
            adr += 1
            k = model.dof_parentid[k]
    model.nM = adr

    # ---- geoms -----------------------------------------------------------
    geoms = dict(names=[], type=[], bodyid=[], pos=[], quat=[], size=[], friction=[],
                 solref=[], solimp=[], solmix=[], margin=[], gap=[], contype=[],
                 conaffinity=[], condim=[], priority=[])

    def add_geom(g, bodyid, off_pos, off_quat):
        contype = int(g.get('contype', 1))
        conaffinity = g.get('conaffinity', '1')
        conaffinity = int(_bool(conaffinity)) if conaffinity.lower() in ('true', 'false') else int(conaffinity)
        if contype == 0 and conaffinity == 0:
            return  # visual geom (mjcf.py:247-249); irrelevant to the hot path
        gtype = g.get('type', 'sphere')
        if gtype not in GEOM_TYPES:
            raise NotImplementedError(f'geom type {gtype}')
        pos = _floats(g.get('pos'), 3, [0, 0, 0])
        if g.get('euler') is not None:
            quat = euler_xyz2quat(_floats(g.get('euler'), 3))
        else:
            quat = _floats(g.get('quat'), 4, [1, 0, 0, 0])
        quat = quat/np.linalg.norm(quat)
        size = np.zeros(3)
        raw_size = _floats(g.get('size'), None, [0])
        size[:min(3, len(raw_size))] = raw_size[:3]
        if g.get('fromto') is not None:
            ft = _floats(g.get('fromto'), 6)
            vec = ft[3:] - ft[:3]
            length = np.linalg.norm(vec)
            pos = 0.5*(ft[:3] + ft[3:])
            zaxis = vec/length
            ref = np.array([0., 0, 1])
            cross = np.cross(ref, zaxis)
            s = np.linalg.norm(cross)
            ang = np.arctan2(s, ref @ zaxis)
            quat = axisangle2quat(cross/s, ang) if s > 1e-12 else (
                np.array([1., 0, 0, 0]) if zaxis[2] > 0 else np.array([0., 1, 0, 0]))
            size[1] = 0.5*length
        geoms['names'].append(g.get('name', f'_anon_geom_{len(geoms["names"])}'))
        geoms['type'].append(GEOM_TYPES[gtype])
        geoms['bodyid'].append(bodyid)
        geoms['pos'].append(off_pos + quat2mat(off_quat) @ pos)
        geoms['quat'].append(quat_mul(off_quat, quat))
        geoms['size'].append(size)
        geoms['friction'].append(_floats(g.get('friction'), 3, [1, 0.005, 0.0001]))
        geoms['solref'].append(_floats(g.get('solref'), 2, DEFAULT_SOLREF))
        geoms['solimp'].append(_floats(g.get('solimp'), 5, DEFAULT_SOLIMP))
        geoms['solmix'].append(float(g.get('solmix', 1)))
        geoms['margin'].append(float(g.get('margin', 0)))
        geoms['gap'].append(float(g.get('gap', 0)))
        geoms['contype'].append(contype)
        geoms['conaffinity'].append(conaffinity)
        geoms['condim'].append(int(g.get('condim', 3)))
        geoms['priority'].append(int(g.get('priority', 0)))

    for g, pos, quat in world_geoms:
        add_geom(g, 0, pos, quat)
    for i, body in enumerate(kept):
        if i == 0:
            continue
        for g in body.geoms:
            add_geom(g, i, np.zeros(3), np.array([1., 0, 0, 0]))
    model.geom_names = geoms['names']
    ng = len(geoms['names'])
    model.geom_type = np.array(geoms['type'], dtype=np.int32)
    model.geom_bodyid = np.array(geoms['bodyid'], dtype=np.int32)
    model.geom_pos = np.array(geoms['pos'], dtype=float).reshape(ng, 3)
    model.geom_quat = np.array(geoms['quat'], dtype=float).reshape(ng, 4)
    model.geom_size = np.array(geoms['size'], dtype=float).reshape(ng, 3)
    model.geom_friction = np.array(geoms['friction'], dtype=float).reshape(ng, 3)
    model.geom_solref = np.array(geoms['solref'], dtype=float).reshape(ng, 2)
    model.geom_solimp = np.array(geoms['solimp'], dtype=float).reshape(ng, 5)
    model.geom_solmix = np.array(geoms['solmix'], dtype=float)
    model.geom_margin = np.array(geoms['margin'], dtype=float)
    model.geom_gap = np.array(geoms['gap'], dtype=float)
    model.geom_contype = np.array(geoms['contype'], dtype=np.int32)
    model.geom_conaffinity = np.array(geoms['conaffinity'], dtype=np.int32)
    model.geom_condim = np.array(geoms['condim'], dtype=np.int32)
    model.geom_priority = np.array(geoms['priority'], dtype=np.int32)
    rbound = np.zeros(ng)
    for g in range(ng):
        t, s = model.geom_type[g], model.geom_size[g]
        if t == GEOM_SPHERE:
            rbound[g] = s[0]
        elif t == GEOM_CAPSULE:
            rbound[g] = s[0] + s[1]
        elif t == GEOM_CYLINDER:
            rbound[g] = np.hypot(s[0], s[1])
        elif t in (GEOM_BOX, GEOM_ELLIPSOID):
            rbound[g] = np.linalg.norm(s) if t == GEOM_BOX else s.max()
        else:
            rbound[g] = 0.0  # plane / hfield / mesh
    model.geom_rbound = rbound

    # ---- actuators -------------------------------------------------------
    act = dict(names=[], kind=[], trnid=[], gain=[], bias=[], ctrllimited=[], ctrlrange=[],
               forcelimited=[], forcerange=[], gear=[])
    act_root = root.find('actuator')
    if act_root is not None:
        for a in act_root:
            if a.tag not in ('position', 'velocity', 'motor'):
                raise NotImplementedError(
                    f'actuator <{a.tag}> (muscles/tendons are out of scope, SURVEY.md section 2 row 4)')
            jname = a.get('joint')
            jid = model.jnt_names.index(jname)
            if model.jnt_type[jid] not in (JNT_HINGE, JNT_SLIDE):
                raise ValueError('actuated joint must be hinge/slide (mjcf.py:809-813)')
            act['names'].append(a.get('name'))
            act['trnid'].append(jid)
            if a.tag == 'position':
                kp = float(a.get('kp', 1))
                kv = float(a.get('kv', 0))
                act['kind'].append(ACT_POSITION)
                act['gain'].append([kp, 0, 0])
                act['bias'].append([0, -kp, -kv])
            elif a.tag == 'velocity':
                kv = float(a.get('kv', 1))
                act['kind'].append(ACT_VELOCITY)
                act['gain'].append([kv, 0, 0])
                act['bias'].append([0, 0, -kv])
            else:
                act['kind'].append(ACT_MOTOR)
                act['gain'].append([1, 0, 0])
                act['bias'].append([0, 0, 0])
            crange = _floats(a.get('ctrlrange'), 2, [0, 0])
            frange = _floats(a.get('forcerange'), 2, [0, 0])
            climited = a.get('ctrllimited')
            flimited = a.get('forcelimited')
            act['ctrllimited'].append(
                bool(crange[0] != 0 or crange[1] != 0)
                if climited is None or climited == 'auto' else _bool(climited))
            act['forcelimited'].append(
                bool(frange[0] != 0 or frange[1] != 0)
                if flimited is None or flimited == 'auto' else _bool(flimited))
            act['ctrlrange'].append(crange)
            act['forcerange'].append(frange)
            gear = _floats(a.get('gear'), None, [1])
            act['gear'].append(float(gear[0]))
    nu = len(act['names'])
    model.actuator_names = act['names']
    model.actuator_kind = np.array(act['kind'], dtype=np.int32)
    model.actuator_trnid = np.array(act['trnid'], dtype=np.int32)
    model.actuator_trntype = np.zeros(nu, dtype=np.int32)
    model.actuator_gainprm = np.array(act['gain'], dtype=float).reshape(nu, 3)
    model.actuator_biasprm = np.array(act['bias'], dtype=float).reshape(nu, 3)
    model.actuator_ctrllimited = np.array(act['ctrllimited'], dtype=np.int32)
    model.actuator_ctrlrange = np.array(act['ctrlrange'], dtype=float).reshape(nu, 2)
    model.actuator_forcelimited = np.array(act['forcelimited'], dtype=np.int32)
    model.actuator_forcerange = np.array(act['forcerange'], dtype=float).reshape(nu, 2)
    model.actuator_gear = np.array(act['gear'], dtype=float)

    # ---- sensors ---------------------------------------------------------
    sens = dict(names=[], type=[], objid=[], adr=[], dim=[])
    adr = 0
    if sensor_root is not None:
        for s in sensor_root:
            if s.tag not in SENSOR_TYPES:
                raise NotImplementedError(f'sensor <{s.tag}> is outside the hot path')
            stype, dim = SENSOR_TYPES[s.tag]
            if stype in (SENS_FRAMEPOS, SENS_FRAMEQUAT, SENS_FRAMELINVEL, SENS_FRAMEANGVEL):
                if s.get('objtype', 'body') != 'body':
                    raise NotImplementedError('frame sensors: objtype=body only (mjcf.py:958-976)')
                objid = model.body_names.index(s.get('objname'))
            elif stype in (SENS_JOINTPOS, SENS_JOINTVEL, SENS_JOINTLIMITFRC):
                objid = model.jnt_names.index(s.get('joint'))
            else:
                objid = model.actuator_names.index(s.get('actuator'))
            sens['names'].append(s.get('name'))
            sens['type'].append(stype)
            sens['objid'].append(objid)
            sens['adr'].append(adr)
            sens['dim'].append(dim)
            adr += dim
    model.sensor_names = sens['names']
    model.sensor_type = np.array(sens['type'], dtype=np.int32)
    model.sensor_objid = np.array(sens['objid'], dtype=np.int32)
    model.sensor_adr = np.array(sens['adr'], dtype=np.int32)
    model.sensor_dim = np.array(sens['dim'], dtype=np.int32)
    model.nsensordata = adr

    # ---- keyframe --------------------------------------------------------
    model.key_qpos = model.qpos0.copy()
    model.key_qvel = np.zeros(nv)
    model.key_ctrl = np.zeros(nu)
    keyframe = root.find('keyframe')
    if keyframe is not None and len(keyframe):
        key = keyframe[0]
        if key.get('qpos') is not None:
            model.key_qpos = _floats(key.get('qpos'), nq)
        if key.get('qvel') is not None:
            model.key_qvel = _floats(key.get('qvel'), nv)
        if key.get('ctrl') is not None:
            model.key_ctrl = _floats(key.get('ctrl'), nu)

    pairs = []
    if root.find('contact') is not None:
        for elem in root.find('contact'):
            if elem.tag != 'pair':
                raise NotImplementedError(f'<contact><{elem.tag}> is outside the batched path')
            pairs.append(elem)

    _compile_collision_candidates(model, pairs, frictionless_pairs)
    _compile_invweight0(model)
    return model


# --------------------------------------------------------------------------
# Compile-time numerics
# --------------------------------------------------------------------------

def _mix_friction(priority1, priority2, friction1, friction2):
    """mj_contactParam's friction of a geom pair: the higher-priority geom's, else the larger of the
    two, floored at MJ_MINMU, element-wise (arrays broadcast).  The one copy of the rule: the compiler
    (_mix_contact_params) and the per-environment tables (candidate_friction) both call it."""
    return np.maximum(MJ_MINMU, np.where(priority1 > priority2, friction1,
                                         np.where(priority2 > priority1, friction2, np.maximum(friction1, friction2))))


def _mix_contact_params(model, g1, g2):
    """mj_contactParam for equal priorities (SURVEY.md Appendix A.6)."""
    p1, p2 = model.geom_priority[g1], model.geom_priority[g2]
    friction = _mix_friction(p1, p2, model.geom_friction[g1], model.geom_friction[g2])
    if p1 != p2:
        g = g1 if p1 > p2 else g2
        return friction, model.geom_solref[g].copy(), model.geom_solimp[g].copy()
    m1, m2 = model.geom_solmix[g1], model.geom_solmix[g2]
    if m1 >= MJ_MINVAL and m2 >= MJ_MINVAL:
        mix = m1/(m1 + m2)
    elif m1 < MJ_MINVAL and m2 < MJ_MINVAL:
        mix = 0.5
    elif m1 < MJ_MINVAL:
        mix = 0.0
    else:
        mix = 1.0
    r1, r2 = model.geom_solref[g1], model.geom_solref[g2]
    if r1[0] > 0 and r2[0] > 0:
        solref = mix*r1 + (1 - mix)*r2
    else:
        solref = np.minimum(r1, r2)
    solimp = mix*model.geom_solimp[g1] + (1 - mix)*model.geom_solimp[g2]
    return friction, solref, solimp


PAIR_MIN_FRICTION = 0.1


def _compile_pair_candidates(model, pairs, frictionless_pairs='refuse'):
    """Explicit ``<contact><pair>`` self-collisions (mjcf.py:1012-1033: one pair per couple of
    collision geoms of the two links, ``condim=3``, ``friction=[0]*5``, optionally ``solref``).
    Sphere-sphere only (candidate kind 20, ``mjc_SphereSphere``; kind 21 for a pair at the friction
    floor under ``frictionless_pairs='hard'``: the same geometry and parameters, solved as one hard
    normal row per contact).  An explicit pair bypasses the
    contype / conaffinity and same-body / parent-child filters; attributes the element does not
    give come from the two geoms by the mixing rule, as MuJoCo's compiler fills them in."""
    cands = []
    for elem in pairs:
        names = [elem.get('geom1'), elem.get('geom2')]
        for name in names:
            if name not in model.geom_names:
                raise ValueError(f'<pair>: unknown geom "{name}"')
        g1, g2 = (model.geom_names.index(name) for name in names)
        if model.geom_bodyid[g1] == 0 or model.geom_bodyid[g2] == 0:
            raise NotImplementedError('<pair> with a world geom: use contype / conaffinity')
        if model.geom_bodyid[g1] == model.geom_bodyid[g2]:
            raise ValueError(f'<pair> {names}: both geoms on one body')
        if model.geom_type[g1] != GEOM_SPHERE or model.geom_type[g2] != GEOM_SPHERE:
            raise NotImplementedError(
                f'<pair> {names}: only sphere-sphere self-collisions in this round (capsule pairs need mjc_CapsuleCapsule)')
        if int(elem.get('condim', 3)) != 3:
            raise NotImplementedError('condim must be 3 (mjcf.py:1029)')
        friction, solref, solimp = _mix_contact_params(model, g1, g2)
        if elem.get('friction') is not None:
            given = _floats(elem.get('friction'))
            if len(given) > 1 and given[1] != given[0]:
                raise NotImplementedError('<pair> friction: the two tangential coefficients must be equal')
            friction = [given[0]]
        if elem.get('solref') is not None:
            solref = _floats(elem.get('solref'), 2)
        if elem.get('solimp') is not None:
            given = _floats(elem.get('solimp'))
            solimp = np.concatenate([given, np.array([0.9, 0.95, 0.001, 0.5, 2.0])[len(given):]])
        margin = float(elem.get('margin')) if elem.get('margin') is not None else max(model.geom_margin[g1], model.geom_margin[g2])
        gap = float(elem.get('gap')) if elem.get('gap') is not None else max(model.geom_gap[g1], model.geom_gap[g2])
        if friction[0] <= MJ_MINMU and frictionless_pairs == 'hard':
            # One hard row n.J.qacc >= aref per contact with the normal force as a multiplier
            # (fb_device.h): drops the 1e-5 n of tangential force such a cone carries and the
            # O(mu) softness of its normal.  mu stays at the floor for the record.
            cands.append((g1, g2, 21, MJ_MINMU, solref, solimp, margin, gap))
            continue
        if friction[0] < PAIR_MIN_FRICTION:
            # A pyramidal contact's rows carry D = 1/(2 mu^2 R) (mj_makeImpedance): at the floor
            # mu = 1e-5 that the reference's friction=[0]*5 pairs get (mjcf.py:1029), the normal
            # direction is 1e10 times stiffer than at mu = 1 and its residual J.qacc - aref has to
            # be resolved to 1e-11 relative -- out of reach of the fp32 primal Newton step
            # (DESIGN.md section 8).
            hint = (" parse_mjcf(..., frictionless_pairs='hard') solves frictionless pairs as hard normal rows"
                    if friction[0] <= MJ_MINMU else '')
            raise NotImplementedError(
                f'<pair> {names}: friction {friction[0]:g} < {PAIR_MIN_FRICTION}: near-frictionless pyramidal '
                f'contacts are too stiff for the fp32 solver (DESIGN.md section 8).{hint}')
        cands.append((g1, g2, 20, max(MJ_MINMU, friction[0]), solref, solimp, margin, gap))
    return cands


def _compile_collision_candidates(model, pairs=(), frictionless_pairs='refuse'):
    """Enumerate plane-vs-{sphere, capsule end, box corner, ellipsoid} candidates (and the four points of a cylinder) with mixed parameters.

    Pair filter ``(contype1 & conaffinity2) || (contype2 & conaffinity1)``,
    same-body pairs skipped; the world's planes against tree geoms is what the
    builder's contype/conaffinity choice leaves (mjcf.py:254-255, 1203).
    geom1 is the plane (lower geom type).  Order: by geom2 id, then plane id,
    capsule + end before - end.
    """
    cands = []
    for g2 in range(model.ngeom):
        if model.geom_bodyid[g2] == 0:
            continue
        for g1 in range(model.ngeom):
            if model.geom_bodyid[g1] != 0:
                continue
            hit = ((model.geom_contype[g1] & model.geom_conaffinity[g2])
                   or (model.geom_contype[g2] & model.geom_conaffinity[g1]))
            if not hit:
                continue
            if model.geom_type[g1] != GEOM_PLANE:
                raise NotImplementedError(
                    f'arena geom "{model.geom_names[g1]}": only planes collide in this round')
            if model.geom_type[g2] not in (GEOM_SPHERE, GEOM_CAPSULE, GEOM_BOX, GEOM_ELLIPSOID, GEOM_CYLINDER):
                raise NotImplementedError(
                    f'geom "{model.geom_names[g2]}": only sphere/capsule/box/ellipsoid/cylinder vs plane in this round')
            if max(model.geom_condim[g1], model.geom_condim[g2]) != 3:
                raise NotImplementedError('condim must be 3 (mjcf.py:256)')
            friction, solref, solimp = _mix_contact_params(model, g1, g2)
            margin = max(model.geom_margin[g1], model.geom_margin[g2])
            gap = max(model.geom_gap[g1], model.geom_gap[g2])
            # plane-box (mjc_PlaneBox): the eight corners in bit order, x fastest
            # plane-ellipsoid (mjc_PlaneConvex with the ellipsoid's support function): one candidate, 10
            # plane-cylinder (mjc_PlaneCylinder): lowest rim point, the rim point at the other end, and
            # the two triangle points on the lower rim: 11 .. 14
            ends = {GEOM_SPHERE: [0], GEOM_CAPSULE: [1, -1], GEOM_BOX: list(range(2, 10)), GEOM_ELLIPSOID: [10],
                    GEOM_CYLINDER: [11, 12, 13, 14]}[int(model.geom_type[g2])]
            for end in ends:
                cands.append((g1, g2, end, float(friction[0]), solref, solimp, margin, gap))
    # explicit pairs come last (MuJoCo's broad phase lists them ahead of the filtered ones; the
    # order of the contacts does not enter the solution, only the order of the rows)
    cands += _compile_pair_candidates(model, pairs, frictionless_pairs)
    n = len(cands)
    model.cand_geom1 = np.array([c[0] for c in cands], dtype=np.int32)
    model.cand_geom2 = np.array([c[1] for c in cands], dtype=np.int32)
    model.cand_end = np.array([c[2] for c in cands], dtype=np.int32)
    model.cand_friction = np.array([c[3] for c in cands], dtype=float)
    model.cand_solref = np.array([c[4] for c in cands], dtype=float).reshape(n, 2)
    model.cand_solimp = np.array([c[5] for c in cands], dtype=float).reshape(n, 5)
    model.cand_margin = np.array([c[6] for c in cands], dtype=float)
    model.cand_gap = np.array([c[7] for c in cands], dtype=float)


def candidate_friction(model, geom_friction):
    """The mixed sliding friction of every collision candidate, ``[..., ncand]``, for the sliding
    frictions ``geom_friction [..., ngeom]`` (``model.geom_friction[:, 0]`` edited): what
    ``parse_mjcf`` compiles into ``cand_friction`` for a model with those frictions -- the
    candidate's two geoms mixed by priority or max, floored at ``MJ_MINMU``.  Explicit ``<pair>``
    candidates (kinds 20 and 21) keep the model's value: a pair takes its friction from the pair
    element."""
    geom_friction = np.asarray(geom_friction, dtype=np.float64)
    g1, g2 = model.cand_geom1, model.cand_geom2
    mixed = _mix_friction(model.geom_priority[g1], model.geom_priority[g2], geom_friction[..., g1], geom_friction[..., g2])
    pair = (model.cand_end == 20) | (model.cand_end == 21)
    return np.where(pair, model.cand_friction, mixed)


def soft_pair_model(model):
    """The model as MuJoCo solves it: a copy whose hard frictionless pairs (kind 21) are the soft
    pyramidal pairs (kind 20, mu at the floor) the reference writes.  This is what a
    double-precision reference solver takes to check the hard rows against."""
    out = copy.copy(model)
    out.cand_end = np.where(model.cand_end == 21, 20, model.cand_end).astype(np.int32)
    return out


def forward_kinematics(model, qpos):
    """Body frames at ``qpos`` (fp64 NumPy; compile-time use and tests).

    Follows SURVEY.md Appendix A.1.  Returns a dict of arrays.
    """
    nb = model.nbody
    xpos = np.zeros((nb, 3))
    xquat = np.tile([1., 0, 0, 0], (nb, 1))
    xanchor = np.zeros((model.njnt, 3))
    xaxis = np.zeros((model.njnt, 3))
    for b in range(1, nb):
        p = model.body_parentid[b]
        jid = model.body_jntid[b]
        if jid >= 0 and model.jnt_type[jid] == JNT_FREE:
            adr = model.jnt_qposadr[jid]
            pos = qpos[adr:adr+3].copy()
            quat = qpos[adr+3:adr+7]/np.linalg.norm(qpos[adr+3:adr+7])
            xanchor[jid] = pos
            xaxis[jid] = [0, 0, 1]
        else:
            pos = xpos[p] + quat2mat(xquat[p]) @ model.body_pos[b]
            quat = quat_mul(xquat[p], model.body_quat[b])
            if jid >= 0:
                adr = model.jnt_qposadr[jid]
                rot = quat2mat(quat)
                xanchor[jid] = pos + rot @ model.jnt_pos[jid]
                xaxis[jid] = rot @ model.jnt_axis[jid]
                if model.jnt_type[jid] == JNT_HINGE:
                    quat = quat_mul(quat, axisangle2quat(model.jnt_axis[jid], qpos[adr] - model.qpos0[adr]))
                    pos = xanchor[jid] - quat2mat(quat) @ model.jnt_pos[jid]
                else:
                    pos = pos + xaxis[jid]*(qpos[adr] - model.qpos0[adr])
        quat = quat/np.linalg.norm(quat)
        xpos[b] = pos
        xquat[b] = quat
    xmat = np.array([quat2mat(q) for q in xquat])
    xipos = xpos + np.einsum('bij,bj->bi', xmat, model.body_ipos)
    ximat = np.array([xmat[b] @ quat2mat(model.body_iquat[b]) for b in range(nb)])
    return dict(xpos=xpos, xquat=xquat, xmat=xmat, xipos=xipos, ximat=ximat,
                xanchor=xanchor, xaxis=xaxis)


def body_jacobian(model, kin, body, point):
    """Translational / rotational Jacobian (3 x nv each) of ``point`` on ``body``."""
    jacp = np.zeros((3, model.nv))
    jacr = np.zeros((3, model.nv))
    b = body
    while b > 0:
        jid = model.body_jntid[b]
        if jid >= 0:
            adr = model.jnt_dofadr[jid]
            if model.jnt_type[jid] == JNT_FREE:
                rot = kin['xmat'][b]
                for k in range(3):
                    jacp[k, adr+k] = 1.0
                    axis = rot[:, k]
                    jacr[:, adr+3+k] = axis
                    jacp[:, adr+3+k] = np.cross(axis, point - kin['xpos'][b])
            elif model.jnt_type[jid] == JNT_HINGE:
                axis = kin['xaxis'][jid]
                jacr[:, adr] = axis
                jacp[:, adr] = np.cross(axis, point - kin['xanchor'][jid])
            else:
                jacp[:, adr] = kin['xaxis'][jid]
        b = model.body_parentid[b]
    return jacp, jacr


def dense_mass_matrix(model, qpos):
    """M(q) = sum_b m Jp^T Jp + Jr^T I Jr (+ armature) -- O(n^2) definition."""
    kin = forward_kinematics(model, qpos)
    mass = np.zeros((model.nv, model.nv))
    for b in range(1, model.nbody):
        if model.body_mass[b] == 0 and not model.body_inertia[b].any():
            continue
        jacp, jacr = body_jacobian(model, kin, b, kin['xipos'][b])
        inertia = kin['ximat'][b] @ np.diag(model.body_inertia[b]) @ kin['ximat'][b].T
        mass += model.body_mass[b]*jacp.T @ jacp + jacr.T @ inertia @ jacr
    mass += np.diag(model.dof_armature)
    return mass, kin


def _compile_invweight0(model):
    """dof_invweight0 / body_invweight0 / meaninertia at qpos0 (Appendix A.9)."""
    nv = model.nv
    model.body_invweight0 = np.zeros((model.nbody, 2))
    model.dof_invweight0 = np.zeros(nv)
    if nv == 0:
        return
    mass, kin = dense_mass_matrix(model, model.qpos0)
    minv = np.linalg.inv(mass)
    model.meaninertia = float(np.mean(np.diag(mass)))
    diag = np.diag(minv).copy()
    for jid in range(model.njnt):
        adr = model.jnt_dofadr[jid]
        if model.jnt_type[jid] == JNT_FREE:
            diag[adr:adr+3] = diag[adr:adr+3].mean()
            diag[adr+3:adr+6] = diag[adr+3:adr+6].mean()
    model.dof_invweight0 = np.maximum(diag, MJ_MINVAL)
    for b in range(1, model.nbody):
        if model.body_dofadr[b] < 0 and not _has_moving_ancestor(model, b):
            continue
        jacp, jacr = body_jacobian(model, kin, b, kin['xipos'][b])
        ap = jacp @ minv @ jacp.T
        ar = jacr @ minv @ jacr.T
        model.body_invweight0[b, 0] = max(np.trace(ap)/3, MJ_MINVAL)
        model.body_invweight0[b, 1] = max(np.trace(ar)/3, MJ_MINVAL)


def _has_moving_ancestor(model, body):
    b = body
    while b > 0:
        if model.body_jntid[b] >= 0:
            return True
        b = model.body_parentid[b]
    return False
