"""ctypes wrapper of the CPU oracle (oracle/_build/liborc.so).  TEST INFRASTRUCTURE ONLY:
imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from rapier_b200 import _abi as A
from rapier_b200.sets import as_array

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "_build", "liborc.so")


def build():
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR])


_libs = {}


def lib(fast=False):
    """fast=False: the bit-exact oracle (the parity checker).  fast=True: the CPU-baseline build of the same sources
    (-O3 -march=native, built by this process into a temporary directory that is removed when it exits: the binary
    only fits this host, and bench.py must leave the tree untouched; bench.py's cpu_baseline / --impl reference legs)."""
    if fast not in _libs:
        path = LIB_PATH
        if fast:
            out = tempfile.mkdtemp(prefix="rapier_b200_oracle_fast_")
            atexit.register(shutil.rmtree, out, True)
            path = os.path.join(out, "liborc_fast.so")
            subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "fast", f"FAST_DIR={out}"])
        elif not os.path.exists(LIB_PATH):
            build()
        L = C.CDLL(path)
        L.orc_world_create.restype = C.c_void_p
        L.orc_world_create.argtypes = [C.POINTER(A.RbIntegrationParameters)]
        L.orc_world_destroy.argtypes = [C.c_void_p]
        L.orc_world_set_scene.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_world_set_params.argtypes = [C.c_void_p, C.POINTER(A.RbIntegrationParameters)]
        L.orc_world_step.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.c_int32]
        L.orc_world_get_body_states.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_world_set_body_states.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_world_num_bodies.argtypes = [C.c_void_p]
        L.orc_world_get_counters.argtypes = [C.c_void_p, C.POINTER(A.RbCounters)]
        L.orc_world_get_contact_pairs.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_world_debug_read.restype = C.c_int64
        L.orc_world_debug_read.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]
        L.orc_set_threads.argtypes = [C.c_int]
        L.orc_contact_manifold.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float,
                                           C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_world_insert.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_world_remove_bodies.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_world_insert_joints.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_world_remove_joints.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_world_update_joints.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32]
        L.orc_world_get_quarantine.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
        L.orc_world_get_sleeping.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_world_wake_up.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_world_set_body_forces.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_world_set_next_kinematic_positions.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        L.orc_world_drain_collision_events.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_world_drain_contact_force_events.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
        L.orc_kat.argtypes = [C.c_char_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]
        L.orc_world_add_hull.restype = C.c_int32
        L.orc_world_add_hull.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
        _libs[fast] = L
    return _libs[fast]


class OracleWorld:
    """Same surface as rapier_b200.PhysicsWorld, backed by the CPU oracle."""

    def __init__(self, scene, params=None, threads=1, fast=False):
        self.L = lib(fast)
        self.params = params or A.RbIntegrationParameters.default()
        self.h = self.L.orc_world_create(C.byref(self.params))
        self.gravity = scene.gravity
        self.L.orc_set_threads(threads)
        nb, nc, nj = len(scene.bodies), len(scene.colliders), len(scene.joints)
        self._nhulls = 0
        self.sync_hulls(scene.colliders)
        self._b = as_array(scene.bodies.descs, A.RbBodyDesc)
        self._c = as_array(scene.colliders.descs, A.RbColliderDesc)
        self._j = as_array(scene.joints.descs, A.RbJointDesc)
        rc = self.L.orc_world_set_scene(self.h, nb, self._b, nc, self._c, nj, self._j)
        if rc != 0:
            raise RuntimeError(f"orc_world_set_scene failed: {rc}")
        self.nb = nb

    def __del__(self):
        try:
            self.L.orc_world_destroy(self.h)
        except Exception:
            pass

    def sync_hulls(self, colliders):
        from rapier_b200.sets import hull_arrays
        for k in range(self._nhulls, len(getattr(colliders, "hulls", []))):
            verts, sizes, idx = hull_arrays(colliders.hulls[k])
            hid = self.L.orc_world_add_hull(self.h, len(verts), verts.ctypes.data, len(sizes), sizes.ctypes.data, idx.ctypes.data)
            assert hid == k + 1, (hid, k)
            self._nhulls = k + 1

    def step(self, n=1):
        g = (C.c_float * 3)(*self.gravity)
        rc = self.L.orc_world_step(self.h, g, n)
        assert rc == 0

    def insert(self, body_descs, collider_descs):
        """Mirror of PhysicsPipeline.insert (appended bodies / colliders)."""
        b = as_array(body_descs, A.RbBodyDesc)
        c = as_array(collider_descs, A.RbColliderDesc)
        rc = self.L.orc_world_insert(self.h, len(body_descs), b, len(collider_descs), c)
        assert rc == 0, rc
        self.nb += len(body_descs)

    def insert_joints(self, joint_descs):
        """Mirror of PhysicsPipeline.insert_joints (appended joints)."""
        j = as_array(joint_descs, A.RbJointDesc)
        rc = self.L.orc_world_insert_joints(self.h, len(joint_descs), j)
        assert rc == 0, rc

    def remove_joints(self, indices):
        idx = np.ascontiguousarray(indices, np.int32)
        rc = self.L.orc_world_remove_joints(self.h, len(idx), idx.ctypes.data)
        assert rc == 0, rc

    def update_joints(self, indices, joint_descs, wake_up=True):
        idx = np.ascontiguousarray(indices, np.int32)
        j = as_array(joint_descs, A.RbJointDesc)
        rc = self.L.orc_world_update_joints(self.h, len(idx), idx.ctypes.data, j, 1 if wake_up else 0)
        assert rc == 0, rc

    def quarantine(self):
        n = self.L.orc_world_get_quarantine(self.h, None, 0)
        out = np.zeros(max(n, 1), np.int32)
        if n:
            self.L.orc_world_get_quarantine(self.h, out.ctypes.data, n)
        return out[:n]

    def sleeping(self):
        out = np.zeros(self.nb, np.uint8)
        self.L.orc_world_get_sleeping(self.h, out.ctypes.data)
        return out

    def wake_up(self, indices):
        idx = np.ascontiguousarray(indices, np.int32)
        assert self.L.orc_world_wake_up(self.h, len(idx), idx.ctypes.data) == 0

    def remove_bodies(self, indices):
        idx = np.ascontiguousarray(indices, np.int32)
        rc = self.L.orc_world_remove_bodies(self.h, len(idx), idx.ctypes.data)
        assert rc == 0, rc

    def body_states(self):
        pose = np.zeros((self.nb, 7), np.float32)
        vel = np.zeros((self.nb, 6), np.float32)
        self.L.orc_world_get_body_states(self.h, pose.ctypes.data, vel.ctypes.data)
        return pose, vel

    def set_body_states(self, indices, pose7=None, vel6=None):
        idx = np.ascontiguousarray(indices, np.int32)
        p = None if pose7 is None else np.ascontiguousarray(pose7, np.float32)
        v = None if vel6 is None else np.ascontiguousarray(vel6, np.float32)
        rc = self.L.orc_world_set_body_states(self.h, len(idx), idx.ctypes.data, None if p is None else p.ctypes.data,
                                              None if v is None else v.ctypes.data)
        assert rc == 0

    def counters(self):
        c = A.RbCounters()
        self.L.orc_world_get_counters(self.h, C.byref(c))
        return c.as_dict()

    def set_body_forces(self, indices, force3=None, torque3=None):
        idx = np.ascontiguousarray(indices, np.int32)
        f = None if force3 is None else np.ascontiguousarray(force3, np.float32)
        t = None if torque3 is None else np.ascontiguousarray(torque3, np.float32)
        rc = self.L.orc_world_set_body_forces(self.h, len(idx), idx.ctypes.data, None if f is None else f.ctypes.data,
                                              None if t is None else t.ctypes.data)
        assert rc == 0

    def set_next_kinematic_positions(self, indices, pose7):
        idx = np.ascontiguousarray(indices, np.int32)
        p = np.ascontiguousarray(pose7, np.float32)
        assert self.L.orc_world_set_next_kinematic_positions(self.h, len(idx), idx.ctypes.data, p.ctypes.data) == 0

    def collision_events(self, with_flags=False):
        """Drains the buffered CollisionEvents: list of (collider1, collider2, started, step[, flags])."""
        buf = (A.RbCollisionEvent * 65536)()
        n = self.L.orc_world_drain_collision_events(self.h, 65536, buf)
        if with_flags:
            return [(e.collider1, e.collider2, e.started, e.step, e.flags) for e in buf[:n]]
        return [(e.collider1, e.collider2, e.started, e.step) for e in buf[:n]]

    def contact_force_events(self):
        buf = (A.RbContactForceEvent * 65536)()
        n = self.L.orc_world_drain_contact_force_events(self.h, 65536, buf)
        return [dict(collider1=e.collider1, collider2=e.collider2, total_force=tuple(e.total_force), total_force_magnitude=e.total_force_magnitude,
                     max_force_direction=tuple(e.max_force_direction), max_force_magnitude=e.max_force_magnitude, started=e.started, step=e.step)
                for e in buf[:n]]

    def contact_pairs(self):
        n = self.L.orc_world_get_contact_pairs(self.h, 0, None, None, None, None, None)
        pc = np.zeros((n, 2), np.int32)
        nc = np.zeros(n, np.int32)
        col = np.zeros(n, np.int32)
        nrm = np.zeros((n, 3), np.float32)
        imp = np.zeros((n, 4), np.float32)
        self.L.orc_world_get_contact_pairs(self.h, n, pc.ctypes.data, nc.ctypes.data, col.ctypes.data, nrm.ctypes.data,
                                           imp.ctypes.data)
        return dict(colliders=pc, num_contacts=nc, color=col, normal=nrm, impulses=imp)

    def debug_read(self, table, dtype):
        n = self.L.orc_world_debug_read(self.h, table.encode(), None, 0)
        if n < 0:
            raise KeyError(table)
        buf = np.zeros(n, np.uint8)
        self.L.orc_world_debug_read(self.h, table.encode(), buf.ctypes.data, n)
        return buf.view(dtype)


def contact_manifold(shape1, he1, shape2, he2, t, q, prediction=0.02):
    L = lib()
    he1 = np.asarray(he1, np.float32)
    he2 = np.asarray(he2, np.float32)
    t = np.asarray(t, np.float32)
    q = np.asarray(q, np.float32)
    out = np.zeros((8, 9), np.float32)
    n1 = np.zeros(3, np.float32)
    n2 = np.zeros(3, np.float32)
    n = L.orc_contact_manifold(shape1, he1.ctypes.data, shape2, he2.ctypes.data, t.ctypes.data, q.ctypes.data,
                               C.c_float(prediction), out.ctypes.data, n1.ctypes.data, n2.ctypes.data)
    return out[:n], n1, n2
