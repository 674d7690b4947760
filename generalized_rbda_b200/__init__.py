"""generalized_rbda_b200 — batched ClusterTreeModel dynamics on B200 (sm_100a).

Thin Python binding (ctypes) over the C ABI in include/grbda_cuda.h. PyTorch is used only for
device memory, streams and torch.distributed plumbing; every kernel that runs is one of this
repository's own generated sm_100a kernels inside libgrbda_cuda.so. There is no CPU fallback: if
the shared library has not been built (python -m generalized_rbda_b200.build, or
__graft_entry__.build()) importing this package raises.

The class below mirrors the reference's model API
(reference: include/grbda/Dynamics/ClusterTreeModel.h:23-228, TreeModel.h:15-143) with batched
versions of inverseDynamics / forwardDynamics / getMassMatrix / forwardKinematics.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("GRBDA_LIB_PATH") or os.path.join(_HERE, "libgrbda_cuda.so")  # override: kernel experiments
URDF_DIR = os.path.join(_HERE, "robot-models")

if not os.path.exists(_LIB_PATH):
    raise ImportError(
        "generalized_rbda_b200: %s is missing — build it first "
        "(python -m generalized_rbda_b200.build); there is no CPU fallback" % _LIB_PATH)

os.environ.setdefault("GRBDA_URDF_DIR", URDF_DIR)
_lib = C.CDLL(_LIB_PATH)

ALGO_ID, ALGO_FD, ALGO_FK, ALGO_H, ALGO_PHI = 0, 1, 2, 3, 4
ALGO_NAMES = ["id", "fd", "fk", "h", "phi"]
ALGO_GFA, ALGO_GFS = 5, 6  # tau_in +/- J^T f_ext (external forces on the terminal links)
ALGO_CONTACT_KIN, ALGO_CONTACT_JAC, ALGO_TEST_FORCE, ALGO_OSIM = 8, 9, 10, 11  # operational space (contact points)
ALGO_ID_DERIV, ALGO_FD_DERIV = 12, 13  # derivatives of the dynamics
ALGO_ID_VJP, ALGO_FD_VJP = 14, 15  # vector-Jacobian products of the dynamics (reverse mode)
ALGO_GFA_VJP, ALGO_GFS_VJP, ALGO_CONTACT_KIN_VJP = 16, 17, 18  # ... of the external-force programs, contact kinematics
ALGO_CONTACT_FD, ALGO_CONTACT_IMPULSE = 19, 20  # rigid point contacts: constrained forward dynamics, impulses
PROGRAM_FD_LTL = 7  # dump_program only: forward dynamics as CRBA + bias + sparse L^T D L (kernel variant "ltl")
PROGRAM_INTEGRATE_VJP = -2  # prepare / jit_compile: the reverse integration step (GRBDA_PROGRAM_INTEGRATE_VJP)

_vp = C.c_void_p
_i64 = C.c_int64
_lib.grbda_cuda_last_error_string.restype = C.c_char_p
_lib.grbda_cuda_version.restype = C.c_char_p
_lib.grbda_cuda_model_hash.restype = C.c_uint64
_lib.grbda_cuda_model_hash.argtypes = [_vp]
_lib.grbda_cuda_launch_count.restype = _i64
for _n in ("num_positions", "num_degrees_of_freedom", "num_bodies", "num_clusters"):
    getattr(_lib, "grbda_cuda_" + _n).argtypes = [_vp]
_lib.grbda_cuda_model_create_from_robot.argtypes = [C.c_char_p, C.c_int, C.POINTER(_vp)]
_lib.grbda_cuda_model_create_from_urdf.argtypes = [C.c_char_p, C.c_int, C.POINTER(_vp)]
_lib.grbda_cuda_model_create_from_urdfs.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_int, C.POINTER(_vp)]
_lib.grbda_cuda_model_create.argtypes = [_vp, C.c_int, C.POINTER(_vp)]
_lib.grbda_cuda_describe_urdf.argtypes = [C.POINTER(C.c_char_p), C.c_int, C.c_char_p, _i64, C.POINTER(_i64)]
_lib.grbda_cuda_model_destroy.argtypes = [_vp]
_lib.grbda_cuda_cluster_info.argtypes = [_vp, C.c_int, _vp, _vp]
_lib.grbda_cuda_body_info.argtypes = [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp]
_lib.grbda_cuda_cluster_G.argtypes = [_vp, C.c_int, _vp]
_lib.grbda_cuda_model_gravity.argtypes = [_vp, _vp]
_lib.grbda_cuda_cluster_phi.argtypes = [_vp, C.c_int, _vp, _vp, _vp, _vp]
_lib.grbda_cuda_dump_program.argtypes = [_vp, C.c_int, C.c_char_p, _vp]
_lib.grbda_cuda_kernel_counts.argtypes = [_vp, C.c_int, _vp]
_lib.grbda_cuda_emit_source.argtypes = [_vp, C.c_int, C.c_int, C.c_char_p]
_lib.grbda_cuda_model_prepare.argtypes = [_vp, C.c_int, C.c_int]
_lib.grbda_cuda_kernel_info.argtypes = [_vp, C.c_int, C.c_int, _vp]
_lib.grbda_cuda_jit_compile.argtypes = [_vp, C.c_int, C.c_int, C.c_char_p, C.c_char_p]
for _p in ("f64", "f32"):
    getattr(_lib, "grbda_cuda_inverse_dynamics_" + _p).argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, _vp]
    getattr(_lib, "grbda_cuda_forward_dynamics_" + _p).argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, _vp]
    getattr(_lib, "grbda_cuda_mass_matrix_" + _p).argtypes = [_vp, _vp, _vp, _i64, _vp]
    getattr(_lib, "grbda_cuda_forward_kinematics_" + _p).argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_inverse_dynamics_ext_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_forward_dynamics_ext_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_external_force_bodies.argtypes = [_vp, _vp, _vp]
_lib.grbda_cuda_set_external_force_bodies.argtypes = [_vp, _vp, C.c_int32]
_lib.grbda_cuda_set_contact_points.argtypes = [_vp, C.c_int32, _vp, _vp, _vp]
_lib.grbda_cuda_num_contact_points.argtypes = [_vp]
_lib.grbda_cuda_num_end_effectors.argtypes = [_vp]
_lib.grbda_cuda_contact_kinematics_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_contact_jacobians_f64.argtypes = [_vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_apply_test_force_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_inverse_osim_f64.argtypes = [_vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_inverse_dynamics_derivatives_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_forward_dynamics_derivatives_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_inverse_dynamics_vjp_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_forward_dynamics_vjp_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_inverse_dynamics_ext_vjp_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_forward_dynamics_ext_vjp_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_contact_kinematics_vjp_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_contact_forward_dynamics_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_contact_impulse_f64.argtypes = [_vp, _vp, _vp, _vp, C.c_double, C.c_double, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_integrate_f64.argtypes = [_vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_step_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_integrate_vjp_f64.argtypes = [_vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_step_vjp_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, C.c_double, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64,
                                         _vp]
_lib.grbda_cuda_dynamics_host_f64.argtypes = [_vp, C.c_int, _vp, _vp, _vp, _vp, _i64]
_lib.grbda_cuda_forward_inverse_host_f64.argtypes = [_vp, _vp, _vp, _vp, _vp, _vp, _i64]
_lib.grbda_cuda_bind_host_to_device.argtypes = [C.c_int, _vp]
_lib.grbda_cuda_generate_states.argtypes = [_vp, C.c_uint64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]
_lib.grbda_cuda_constraint_violation_f64.argtypes = [_vp, _vp, _vp, _i64, _vp]
_lib.grbda_cuda_checksum_f64.argtypes = [_vp, _i64, _vp, _vp]
_lib.grbda_cuda_measure_fma_peak.argtypes = [C.c_int, C.c_int, C.c_double, C.POINTER(C.c_double)]

EXPORTED_SYMBOLS = [
    "grbda_cuda_last_error_string", "grbda_cuda_version", "grbda_cuda_model_create",
    "grbda_cuda_model_create_from_urdf", "grbda_cuda_model_create_from_urdfs", "grbda_cuda_describe_urdf", "grbda_cuda_model_create_from_robot", "grbda_cuda_model_destroy",
    "grbda_cuda_num_positions", "grbda_cuda_num_degrees_of_freedom", "grbda_cuda_num_bodies",
    "grbda_cuda_num_clusters", "grbda_cuda_model_hash", "grbda_cuda_cluster_info", "grbda_cuda_body_info",
    "grbda_cuda_cluster_G", "grbda_cuda_model_gravity", "grbda_cuda_cluster_phi", "grbda_cuda_dump_program", "grbda_cuda_kernel_counts", "grbda_cuda_emit_source",
    "grbda_cuda_model_prepare", "grbda_cuda_kernel_info", "grbda_cuda_jit_compile",
    "grbda_cuda_external_force_bodies", "grbda_cuda_inverse_dynamics_ext_f64", "grbda_cuda_forward_dynamics_ext_f64",
    "grbda_cuda_integrate_f64", "grbda_cuda_step_f64", "grbda_cuda_integrate_vjp_f64", "grbda_cuda_step_vjp_f64",
    "grbda_cuda_set_external_force_bodies",
    "grbda_cuda_set_contact_points", "grbda_cuda_num_contact_points", "grbda_cuda_num_end_effectors",
    "grbda_cuda_contact_kinematics_f64", "grbda_cuda_contact_jacobians_f64", "grbda_cuda_apply_test_force_f64",
    "grbda_cuda_inverse_osim_f64",
    "grbda_cuda_inverse_dynamics_derivatives_f64", "grbda_cuda_forward_dynamics_derivatives_f64",
    "grbda_cuda_inverse_dynamics_vjp_f64", "grbda_cuda_forward_dynamics_vjp_f64",
    "grbda_cuda_inverse_dynamics_ext_vjp_f64", "grbda_cuda_forward_dynamics_ext_vjp_f64",
    "grbda_cuda_contact_kinematics_vjp_f64", "grbda_cuda_contact_forward_dynamics_f64", "grbda_cuda_contact_impulse_f64",
    "grbda_cuda_inverse_dynamics_f64", "grbda_cuda_inverse_dynamics_f32",
    "grbda_cuda_forward_dynamics_f64", "grbda_cuda_forward_dynamics_f32",
    "grbda_cuda_mass_matrix_f64", "grbda_cuda_mass_matrix_f32",
    "grbda_cuda_forward_kinematics_f64", "grbda_cuda_forward_kinematics_f32",
    "grbda_cuda_dynamics_host_f64", "grbda_cuda_forward_inverse_host_f64", "grbda_cuda_bind_host_to_device", "grbda_cuda_generate_states", "grbda_cuda_constraint_violation_f64",
    "grbda_cuda_checksum_f64", "grbda_cuda_measure_fma_peak", "grbda_cuda_launch_count",
]

DEFAULT_SEED = 0x6772626461  # "grbda"
# layout of grbda_phi_op (int32 op, a, b; 4 bytes padding; float64 val)
PHI_OP_DTYPE = np.dtype({"names": ["op", "a", "b", "val"], "formats": [np.int32, np.int32, np.int32, np.float64],
                         "offsets": [0, 4, 8, 16], "itemsize": 24})


class _ScheduleStruct(C.Structure):
    """ctypes mirror of grbda_schedule (include/grbda_cuda.h)."""
    _fields_ = [("num_bodies", C.c_int32), ("num_clusters", C.c_int32), ("gravity", C.c_double * 3),
                ("body_parent", _vp), ("body_joint_axis", _vp), ("body_xtree_E", _vp), ("body_xtree_r", _vp),
                ("body_inertia", _vp), ("body_independent", _vp),
                ("cluster_type", _vp), ("cluster_num_bodies", _vp), ("cluster_num_independent", _vp),
                ("cluster_G_offset", _vp), ("G_values", _vp), ("cluster_phi_offset", _vp),
                ("cluster_phi_count", _vp), ("cluster_phi_out_offset", _vp), ("cluster_num_constraints", _vp),
                ("phi_ops", _vp), ("phi_outputs", _vp)]


class Schedule:
    """Flattened structure-of-arrays topology schedule (grbda_schedule) held as numpy arrays: what a
    binding of the reference fills by walking a grbda::ClusterTreeModel (INTEGRATION.md). Every array
    may be edited before ClusterTreeModel.from_schedule(schedule)."""

    FIELDS = (("body_parent", np.int32), ("body_joint_axis", np.int32), ("body_xtree_E", np.float64),
              ("body_xtree_r", np.float64), ("body_inertia", np.float64), ("body_independent", np.uint8),
              ("cluster_type", np.int32), ("cluster_num_bodies", np.int32), ("cluster_num_independent", np.int32),
              ("cluster_G_offset", np.int32), ("G_values", np.float64), ("cluster_phi_offset", np.int32),
              ("cluster_phi_count", np.int32), ("cluster_phi_out_offset", np.int32),
              ("cluster_num_constraints", np.int32), ("phi_ops", PHI_OP_DTYPE), ("phi_outputs", np.int32))

    def __init__(self, gravity=(0.0, 0.0, -9.81)):
        self.gravity = np.array(gravity, dtype=np.float64)
        for name, dt in self.FIELDS:
            setattr(self, name, np.zeros(0, dtype=dt))

    def struct(self):
        """(ctypes struct, keep-alive list): arrays are made contiguous copies of the right dtype."""
        st = _ScheduleStruct()
        st.num_bodies = len(self.body_parent)
        st.num_clusters = len(self.cluster_type)
        st.gravity[:] = [float(x) for x in self.gravity]
        keep = []
        for name, dt in self.FIELDS:
            a = np.ascontiguousarray(getattr(self, name), dtype=dt).reshape(-1)
            if a.size == 0:
                a = np.zeros(1, dtype=dt)  # never hand out a NULL array
            keep.append(a)
            setattr(st, name, a.ctypes.data)
        return st, keep


class GrbdaError(RuntimeError):
    """Raised for every non-zero grbda_status (the reference throws std::runtime_error)."""

    def __init__(self, status, message):
        super().__init__("grbda_cuda status %d: %s" % (status, message))
        self.status = status


def _check(status):
    if status != 0:
        raise GrbdaError(status, _lib.grbda_cuda_last_error_string().decode())


def lib():
    return _lib


def library_path():
    return _LIB_PATH


def launch_count():
    return int(_lib.grbda_cuda_launch_count())


def bind_host_to_device(device=0):
    """CPU affinity + memory policy of the calling thread -> the NUMA node of the GPU's PCIe root."""
    info = (C.c_int32 * 4)()
    _check(_lib.grbda_cuda_bind_host_to_device(device, info))
    return dict(numa_node=info[0], cpus_bound=info[1], mempolicy_set=bool(info[2]), cpus_allowed=info[3])


def measure_fma_peak(device=0, fp32=False, seconds=0.5):
    out = C.c_double()
    _check(_lib.grbda_cuda_measure_fma_peak(device, int(fp32), seconds, C.byref(out)))
    return out.value


def _ptr(t):
    return None if t is None else _vp(t.data_ptr())


def _rows(t, B, n):
    """t as B rows (f_ext [B, nf, 6] -> [B, 6 nf]); n is the row length when there are no rows to infer it from.
    A wrong size is reported by ClusterTreeModel._prep."""
    return t.reshape(B, -1) if B else t.reshape(0, n)


def _stream():
    import torch
    return _vp(torch.cuda.current_stream().cuda_stream)


def describe_urdf(paths):
    """The URDF+ front end's reading of one file or of several files that make one robot (dict: link_order, links
    with parent / children / loop_links / supporting_chain / cluster, clusters)."""
    import json
    if not isinstance(paths, (list, tuple)):
        paths = [paths]
    arr = (C.c_char_p * len(paths))(*[os.fspath(p).encode() for p in paths])
    need = _i64(0)
    _check(_lib.grbda_cuda_describe_urdf(arr, len(paths), None, 0, C.byref(need)))
    buf = C.create_string_buffer(need.value)
    _check(_lib.grbda_cuda_describe_urdf(arr, len(paths), buf, need.value, None))
    return json.loads(buf.value.decode())


class ClusterTreeModel:
    """Batched counterpart of grbda::ClusterTreeModel.

    Construct with from_robot(name) (the reference's robot classes / URDF+ files) or
    from_urdf(path). device=None gives a host-only handle (sizes, topology, emitted programs).
    """

    def __init__(self, handle, device):
        self._h = handle
        self.device = device

    @classmethod
    def from_robot(cls, name, device=0):
        h = _vp()
        _check(_lib.grbda_cuda_model_create_from_robot(name.encode(), -1 if device is None else device, C.byref(h)))
        return cls(h, device)

    @classmethod
    def from_urdf(cls, path, device=0):
        """path: one URDF+ file, or a list of files that together describe one robot (ClusterTreeModel.h:41-53)."""
        h = _vp()
        dev = -1 if device is None else device
        if isinstance(path, (list, tuple)):
            paths = (C.c_char_p * len(path))(*[os.fspath(p).encode() for p in path])
            _check(_lib.grbda_cuda_model_create_from_urdfs(paths, len(path), dev, C.byref(h)))
        else:
            _check(_lib.grbda_cuda_model_create_from_urdf(os.fspath(path).encode(), dev, C.byref(h)))
        return cls(h, device)

    @classmethod
    def from_schedule(cls, schedule, device=0):
        """schedule: a Schedule, or the address of a grbda_schedule struct."""
        h = _vp()
        keep = None
        if isinstance(schedule, Schedule):
            st, keep = schedule.struct()
            schedule = C.addressof(st)
        _check(_lib.grbda_cuda_model_create(schedule, -1 if device is None else device, C.byref(h)))
        del keep
        return cls(h, device)

    def to_schedule(self):
        """The model as a Schedule (numpy arrays), assembled from the introspection entry points."""
        s = Schedule(self.getGravity())
        bodies, clusters = self.bodies(), self.clusters()
        s.body_parent = np.array([b["parent"] for b in bodies], dtype=np.int32)
        s.body_joint_axis = np.array([b["axis"] for b in bodies], dtype=np.int32)
        s.body_xtree_E = np.concatenate([b["E"].reshape(-1) for b in bodies])
        s.body_xtree_r = np.concatenate([b["r"].reshape(-1) for b in bodies])
        s.body_inertia = np.concatenate([b["inertia"].reshape(-1) for b in bodies])
        ind = np.ones(len(bodies), dtype=np.uint8)
        G, ops, outs = [], [], []
        G_off, phi_off, phi_cnt, phi_out_off, ncons = [], [], [], [], []
        n_ops = n_outs = n_G = 0
        for c in clusters:
            G_off.append(n_G), phi_off.append(n_ops), phi_out_off.append(n_outs)
            if c["type"] == 2:
                G.append(c["G"].reshape(-1))
                n_G += c["G"].size
                phi_cnt.append(0)
                ncons.append(c["num_bodies"] - c["num_velocities"])
            elif c["type"] == 3:
                ops.append(c["phi_ops"]), outs.append(c["phi_outputs"])
                n_ops += len(c["phi_ops"])
                n_outs += len(c["phi_outputs"])
                phi_cnt.append(len(c["phi_ops"]))
                ncons.append(len(c["phi_outputs"]))
                ind[c["first_body"]:c["first_body"] + c["num_bodies"]] = c["independent"]
            else:
                phi_cnt.append(0)
                ncons.append(0)
        s.body_independent = ind
        s.cluster_type = np.array([c["type"] for c in clusters], dtype=np.int32)
        s.cluster_num_bodies = np.array([c["num_bodies"] for c in clusters], dtype=np.int32)
        s.cluster_num_independent = np.array([c["num_velocities"] for c in clusters], dtype=np.int32)
        s.cluster_G_offset = np.array(G_off, dtype=np.int32)
        s.G_values = np.concatenate(G) if G else np.zeros(0)
        s.cluster_phi_offset = np.array(phi_off, dtype=np.int32)
        s.cluster_phi_count = np.array(phi_cnt, dtype=np.int32)
        s.cluster_phi_out_offset = np.array(phi_out_off, dtype=np.int32)
        s.cluster_num_constraints = np.array(ncons, dtype=np.int32)
        s.phi_ops = np.concatenate(ops) if ops else np.zeros(0, dtype=PHI_OP_DTYPE)
        s.phi_outputs = np.concatenate(outs) if outs else np.zeros(0, dtype=np.int32)
        return s

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.grbda_cuda_model_destroy(self._h)
            self._h = None

    # ---- sizes / topology (TreeModel.h:25-28) -------------------------------------------------
    def getNumPositions(self):
        return _lib.grbda_cuda_num_positions(self._h)

    def getNumDegreesOfFreedom(self):
        return _lib.grbda_cuda_num_degrees_of_freedom(self._h)

    def getNumBodies(self):
        return _lib.grbda_cuda_num_bodies(self._h)

    def getNumClusters(self):
        return _lib.grbda_cuda_num_clusters(self._h)

    nq = property(getNumPositions)
    nv = property(getNumDegreesOfFreedom)
    nb = property(getNumBodies)
    nc = property(getNumClusters)

    @property
    def hash(self):
        return int(_lib.grbda_cuda_model_hash(self._h))

    def clusters(self):
        out = []
        for c in range(self.nc):
            info = (C.c_int32 * 8)()
            name = C.create_string_buffer(64)
            _check(_lib.grbda_cuda_cluster_info(self._h, c, info, name))
            keys = ("parent", "num_bodies", "num_positions", "num_velocities", "position_index",
                    "velocity_index", "type", "first_body")
            d = dict(zip(keys, list(info)))
            d["joint_type"] = name.value.decode()
            if d["type"] == 2:
                G = np.zeros((d["num_bodies"], d["num_velocities"]))
                _check(_lib.grbda_cuda_cluster_G(self._h, c, G.ctypes.data_as(_vp)))
                d["G"] = G
            elif d["type"] == 3:
                sizes = (C.c_int32 * 2)()
                _check(_lib.grbda_cuda_cluster_phi(self._h, c, None, None, None, sizes))
                ops = np.zeros(sizes[0], dtype=PHI_OP_DTYPE)
                outs = np.zeros(sizes[1], dtype=np.int32)
                ind = np.zeros(d["num_bodies"], dtype=np.uint8)
                _check(_lib.grbda_cuda_cluster_phi(self._h, c, ops.ctypes.data_as(_vp), outs.ctypes.data_as(_vp),
                                                   ind.ctypes.data_as(_vp), sizes))
                d["phi_ops"], d["phi_outputs"], d["independent"] = ops, outs, ind.astype(bool)
            out.append(d)
        return out

    def bodies(self):
        out = []
        for b in range(self.nb):
            info = (C.c_int32 * 4)()
            name = C.create_string_buffer(64)
            E, r, I = np.zeros((3, 3)), np.zeros(3), np.zeros((6, 6))
            _check(_lib.grbda_cuda_body_info(self._h, b, name, info, E.ctypes.data_as(_vp),
                                             r.ctypes.data_as(_vp), I.ctypes.data_as(_vp)))
            out.append(dict(name=name.value.decode(), parent=info[0], cluster=info[1], sub_index=info[2],
                            axis=info[3], E=E, r=r, inertia=I))
        return out

    def getGravity(self):
        g = np.zeros(3)
        _check(_lib.grbda_cuda_model_gravity(self._h, g.ctypes.data_as(_vp)))
        return g

    def dump_program(self, algo, path=None):
        counts = (C.c_int64 * 8)()
        _check(_lib.grbda_cuda_dump_program(self._h, algo, path.encode() if path else None, counts))
        keys = ("nodes", "add", "mul", "div", "sqrt", "sin", "cos", "fusable")
        d = dict(zip(keys, [int(x) for x in counts]))
        d["flops"] = d["add"] + d["mul"] + d["div"] + d["sqrt"]
        return d

    def externalForceBodies(self):
        """Body indices (terminal links) that accept external forces, in the order f_ext uses."""
        n = C.c_int32(0)
        _check(_lib.grbda_cuda_external_force_bodies(self._h, None, C.byref(n)))
        idx = (C.c_int32 * max(1, n.value))()
        _check(_lib.grbda_cuda_external_force_bodies(self._h, idx, C.byref(n)))
        return [int(idx[i]) for i in range(n.value)]

    def setExternalForceBodies(self, bodies):
        """Any distinct body indices (empty: back to the default, the terminal links); the force programs are
        recompiled for the set at run time."""
        arr = (C.c_int32 * max(1, len(bodies)))(*bodies)
        _check(_lib.grbda_cuda_set_external_force_bodies(self._h, arr, len(bodies)))

    def _dynamics_ext(self, name, q, yd, in3, f_ext, out):
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd = self._prep(yd, self.nv, torch.float64)
        in3 = self._prep(in3, self.nv, torch.float64)
        B = q.shape[0]
        nf = len(self.externalForceBodies())
        f_ext = self._prep(_rows(f_ext, B, 6 * nf), 6 * nf, torch.float64)
        if out is None:
            out = torch.empty((B, self.nv), dtype=torch.float64, device=q.device)
        _check(getattr(_lib, name)(self._h, _ptr(q), _ptr(yd), _ptr(in3), _ptr(f_ext), _ptr(out), B, _stream()))
        return out

    def emit_source(self, program, path, park=False):
        """Write the CUDA source the model compiler emits for `program` (constant table + struct Body). park: False,
        True (values parked in the tile rows) or 1 + n (and in a park area of n slots per thread)."""
        _check(_lib.grbda_cuda_emit_source(self._h, program, int(park), path.encode()))

    def kernel_counts(self, algo):
        """Operation counts of the program the default compiled kernel of `algo` runs per state."""
        counts = (C.c_int64 * 8)()
        _check(_lib.grbda_cuda_kernel_counts(self._h, algo, counts))
        keys = ("nodes", "add", "mul", "div", "sqrt", "sin", "cos", "fusable")
        d = dict(zip(keys, [int(x) for x in counts]))
        d["flops"] = d["add"] + d["mul"] + d["div"] + d["sqrt"]
        return d

    # ---- kernel provenance / run-time compilation ------------------------------------------------
    def prepare(self, algo, f32=False):
        """Compile / load the kernels of one entry point now instead of on first use."""
        _check(_lib.grbda_cuda_model_prepare(self._h, algo, int(bool(f32))))

    def kernel_info(self, algo, f32=False):
        info = (C.c_int64 * 8)()
        _check(_lib.grbda_cuda_kernel_info(self._h, algo, int(bool(f32)), info))
        v = [int(x) for x in info]
        return dict(source="jit" if v[0] else "aot", block=v[1], min_blocks=v[2], smem=v[3], program=v[4],
                    parked=bool(v[5] & 1), tma=bool(v[5] & 2), direct=bool(v[5] & 4), from_cache=bool(v[5] & 8),
                    compile_ms=v[6], ready=bool(v[7]))

    def jit_compile(self, algo, f32=False, source_path=None, cubin_path=None):
        """Run-time compiler without a device: CUDA text and / or NVRTC cubin of one entry point (algo -1: generator,
        PROGRAM_INTEGRATE_VJP: the reverse integration step)."""
        _check(_lib.grbda_cuda_jit_compile(self._h, algo, int(bool(f32)),
                                           source_path.encode() if source_path else None,
                                           cubin_path.encode() if cubin_path else None))

    # ---- batched hot path (device tensors) ----------------------------------------------------
    def _prep(self, t, n, dtype=None):
        import torch
        if not t.is_cuda:
            raise ValueError("expected a CUDA tensor")
        if self.device is not None and t.device.index != self.device:
            raise ValueError("tensor lives on cuda:%d but the model was created on cuda:%d" % (t.device.index, self.device))
        if dtype is not None and t.dtype != dtype:
            raise ValueError("dtype mismatch: %s vs %s" % (t.dtype, dtype))
        if t.dtype not in (torch.float64, torch.float32):
            raise ValueError("float64 or float32 tensors are required")
        if t.dim() != 2 or t.shape[1] != n or not t.is_contiguous():
            raise ValueError("expected a contiguous [batch, %d] tensor, got %s" % (n, tuple(t.shape)))
        return t

    def _suffix(self, t):
        import torch
        return "f64" if t.dtype == torch.float64 else "f32"

    def inverseDynamics(self, q, yd, ydd, out=None, f_ext=None):
        """tau[batch, nv] = ID(q, yd, ydd)   (ClusterTreeModel::inverseDynamics). f_ext[batch, nf, 6]:
        world-frame spatial forces on externalForceBodies() (TreeModel::setExternalForces), FP64."""
        import torch
        if f_ext is not None:
            return self._dynamics_ext("grbda_cuda_inverse_dynamics_ext_f64", q, yd, ydd, f_ext, out)
        q = self._prep(q, self.nq)
        yd, ydd = self._prep(yd, self.nv, q.dtype), self._prep(ydd, self.nv, q.dtype)
        if out is None:
            out = torch.empty_like(ydd)
        fn = getattr(_lib, "grbda_cuda_inverse_dynamics_" + self._suffix(q))
        _check(fn(self._h, _ptr(q), _ptr(yd), _ptr(ydd), _ptr(out), q.shape[0], _stream()))
        return out

    def forwardDynamics(self, q, yd, tau, out=None, f_ext=None):
        """ydd[batch, nv] = FD(q, yd, tau)   (ClusterTreeModel::forwardDynamics); f_ext as in inverseDynamics."""
        import torch
        if f_ext is not None:
            return self._dynamics_ext("grbda_cuda_forward_dynamics_ext_f64", q, yd, tau, f_ext, out)
        q = self._prep(q, self.nq)
        yd, tau = self._prep(yd, self.nv, q.dtype), self._prep(tau, self.nv, q.dtype)
        if out is None:
            out = torch.empty_like(tau)
        fn = getattr(_lib, "grbda_cuda_forward_dynamics_" + self._suffix(q))
        _check(fn(self._h, _ptr(q), _ptr(yd), _ptr(tau), _ptr(out), q.shape[0], _stream()))
        return out

    # ---- operational space (contact points) -----------------------------------------------------
    def setContactPoints(self, bodies, offsets, end_effector=None):
        """Contact points: body indices, offsets in the body frames [n, 3], end-effector flags."""
        n = len(bodies)
        b = np.ascontiguousarray(bodies, dtype=np.int32)
        o = np.ascontiguousarray(offsets, dtype=np.float64).reshape(n, 3)
        e = np.ascontiguousarray(end_effector if end_effector is not None else np.zeros(n), dtype=np.uint8)
        _check(_lib.grbda_cuda_set_contact_points(self._h, n, b.ctypes.data_as(_vp), o.ctypes.data_as(_vp),
                                                  e.ctypes.data_as(_vp)))

    @property
    def ncp(self):
        return _lib.grbda_cuda_num_contact_points(self._h)

    @property
    def nee(self):
        return _lib.grbda_cuda_num_end_effectors(self._h)

    def contactKinematics(self, q, yd):
        """(p[batch, n_cp, 3], v[batch, n_cp, 3]): world position / linear velocity of the contact points."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd = self._prep(yd, self.nv, torch.float64)
        p = torch.empty((q.shape[0], self.ncp, 3), dtype=torch.float64, device=q.device)
        v = torch.empty_like(p)
        _check(_lib.grbda_cuda_contact_kinematics_f64(self._h, _ptr(q), _ptr(yd), _ptr(p), _ptr(v), q.shape[0], _stream()))
        return p, v

    def contactJacobians(self, q):
        """J[batch, n_cp, 6, nv], world frame, rows [angular; linear] (contactJacobianWorldFrame)."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        J = torch.empty((q.shape[0], self.ncp, 6, self.nv), dtype=torch.float64, device=q.device)
        _check(_lib.grbda_cuda_contact_jacobians_f64(self._h, _ptr(q), _ptr(J), q.shape[0], _stream()))
        return J

    def applyTestForce(self, q, force):
        """force[batch, n_cp, 3] (world) -> (dstate[batch, n_cp, nv], lambda_inv[batch, n_cp])."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        f = self._prep(force.reshape(q.shape[0], -1), 3 * self.ncp, torch.float64)
        d = torch.empty((q.shape[0], self.ncp, self.nv), dtype=torch.float64, device=q.device)
        lam = torch.empty((q.shape[0], self.ncp), dtype=torch.float64, device=q.device)
        _check(_lib.grbda_cuda_apply_test_force_f64(self._h, _ptr(q), _ptr(f), _ptr(d), _ptr(lam), q.shape[0], _stream()))
        return d, lam

    def inverseOperationalSpaceInertiaMatrix(self, q):
        """Lambda^-1 [batch, 6 n_ee, 6 n_ee] over the end-effectors."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        n = 6 * self.nee
        L = torch.empty((q.shape[0], n, n), dtype=torch.float64, device=q.device)
        _check(_lib.grbda_cuda_inverse_osim_f64(self._h, _ptr(q), _ptr(L), q.shape[0], _stream()))
        return L

    def _active(self, active, B):
        import torch
        if active is None:
            return None
        if not active.is_cuda or active.dtype not in (torch.bool, torch.uint8):
            raise ValueError("active must be a bool or uint8 CUDA tensor")
        if active.dim() != 2 or tuple(active.shape) != (B, self.ncp) or not active.is_contiguous():
            raise ValueError("expected a contiguous [batch, %d] mask, got %s" % (self.ncp, tuple(active.shape)))
        if self.device is not None and active.device.index != self.device:
            raise ValueError("tensor lives on cuda:%d but the model was created on cuda:%d" % (active.device.index, self.device))
        return active

    def contactForwardDynamics(self, q, yd, tau, active=None, damping=0.0):
        """(ydd[batch, nv], lam[batch, n_cp, 3]): forward dynamics with the active contact points held by rigid
        bilateral contacts, lam the world-frame contact forces (include/grbda_cuda.h). active[batch, n_cp] (bool or
        uint8; None: all active) selects the contacts per state; damping >= 0 regularises A (needed when the active
        points are redundant, e.g. two points on one foot)."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd, tau = self._prep(yd, self.nv, torch.float64), self._prep(tau, self.nv, torch.float64)
        B = q.shape[0]
        a = self._active(active, B)
        ydd = torch.empty_like(tau)
        lam = torch.empty((B, self.ncp, 3), dtype=torch.float64, device=q.device)
        _check(_lib.grbda_cuda_contact_forward_dynamics_f64(self._h, _ptr(q), _ptr(yd), _ptr(tau), _ptr(a), float(damping),
                                                            _ptr(ydd), _ptr(lam), B, _stream()))
        return ydd, lam

    def contactImpulse(self, q, yd, active=None, restitution=0.0, damping=0.0):
        """(yd_plus[batch, nv], impulse[batch, n_cp, 3]): the velocity after an impact of the active contact points
        and the world-frame impulses, J_a yd_plus = -restitution J_a yd - damping impulse_a (include/grbda_cuda.h)."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd = self._prep(yd, self.nv, torch.float64)
        B = q.shape[0]
        a = self._active(active, B)
        yd_plus = torch.empty_like(yd)
        imp = torch.empty((B, self.ncp, 3), dtype=torch.float64, device=q.device)
        _check(_lib.grbda_cuda_contact_impulse_f64(self._h, _ptr(q), _ptr(yd), _ptr(a), float(restitution), float(damping),
                                                   _ptr(yd_plus), _ptr(imp), B, _stream()))
        return yd_plus, imp

    def inverseDynamicsDerivatives(self, q, yd, ydd):
        """(dtau_dq, dtau_dyd), each [batch, nv, nv], [b, i, j] = d tau_i / d x_j; dq is the tangent-space
        perturbation of the reference's derivative test (d tau / d ydd is getMassMatrix)."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd, ydd = self._prep(yd, self.nv, torch.float64), self._prep(ydd, self.nv, torch.float64)
        dq = torch.empty((q.shape[0], self.nv, self.nv), dtype=torch.float64, device=q.device)
        dv = torch.empty_like(dq)
        _check(_lib.grbda_cuda_inverse_dynamics_derivatives_f64(self._h, _ptr(q), _ptr(yd), _ptr(ydd), _ptr(dq), _ptr(dv),
                                                                q.shape[0], _stream()))
        return dq.transpose(1, 2), dv.transpose(1, 2)  # the library writes column-major matrices

    def forwardDynamicsDerivatives(self, q, yd, tau):
        """(dydd_dq, dydd_dyd, dydd_dtau), each [batch, nv, nv]; dydd_dtau = H^-1."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd, tau = self._prep(yd, self.nv, torch.float64), self._prep(tau, self.nv, torch.float64)
        dq = torch.empty((q.shape[0], self.nv, self.nv), dtype=torch.float64, device=q.device)
        dv, dt = torch.empty_like(dq), torch.empty_like(dq)
        _check(_lib.grbda_cuda_forward_dynamics_derivatives_f64(self._h, _ptr(q), _ptr(yd), _ptr(tau), _ptr(dq), _ptr(dv),
                                                                _ptr(dt), q.shape[0], _stream()))
        return dq.transpose(1, 2), dv.transpose(1, 2), dt.transpose(1, 2)

    def _vjp(self, dynamics, q, yd, aux, w, f_ext=None):
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd, aux, w = (self._prep(t, self.nv, torch.float64) for t in (yd, aux, w))
        q_bar = torch.empty_like(q)
        yd_bar, aux_bar = torch.empty_like(yd), torch.empty_like(yd)
        B = q.shape[0]
        if f_ext is None:
            _check(getattr(_lib, "grbda_cuda_%s_vjp_f64" % dynamics)(
                self._h, _ptr(q), _ptr(yd), _ptr(aux), _ptr(w), _ptr(q_bar), _ptr(yd_bar), _ptr(aux_bar), B, _stream()))
            return q_bar, yd_bar, aux_bar
        nf6 = 6 * len(self.externalForceBodies())
        f = self._prep(_rows(f_ext, B, nf6), nf6, torch.float64)
        f_bar = torch.empty_like(f)
        _check(getattr(_lib, "grbda_cuda_%s_ext_vjp_f64" % dynamics)(
            self._h, _ptr(q), _ptr(yd), _ptr(aux), _ptr(f), _ptr(w), _ptr(q_bar), _ptr(yd_bar), _ptr(aux_bar),
            _ptr(f_bar), B, _stream()))
        return q_bar, yd_bar, aux_bar, f_bar.reshape(f_ext.shape)

    def inverseDynamicsVJP(self, q, yd, ydd, tau_bar, f_ext=None):
        """(q_bar[batch, nq], yd_bar[batch, nv], ydd_bar[batch, nv]): the cotangent tau_bar of tau = ID(q, yd, ydd)
        pulled back to the inputs (ydd_bar = H tau_bar); q_bar is the gradient with respect to the stored positions.
        With f_ext (as inverseDynamics takes it: tau = ID - J^T f) a fourth tensor, f_bar = -J tau_bar, in the shape
        of f_ext."""
        return self._vjp("inverse_dynamics", q, yd, ydd, tau_bar, f_ext)

    def forwardDynamicsVJP(self, q, yd, tau, ydd_bar, f_ext=None):
        """(q_bar[batch, nq], yd_bar[batch, nv], tau_bar[batch, nv]): the cotangent ydd_bar of ydd = FD(q, yd, tau)
        pulled back to the inputs (tau_bar = H^-1 ydd_bar); q_bar as documented in include/grbda_cuda.h. With f_ext
        (ydd = FD(q, yd, tau + J^T f)) a fourth tensor, f_bar = J tau_bar, in the shape of f_ext."""
        return self._vjp("forward_dynamics", q, yd, tau, ydd_bar, f_ext)

    def contactKinematicsVJP(self, q, yd, p_bar, v_bar):
        """(q_bar[batch, nq], yd_bar[batch, nv]): the cotangents p_bar / v_bar [batch, n_cp, 3] of contactKinematics
        pulled back to the inputs (yd_bar = J_lin^T v_bar); q_bar is the gradient with respect to the stored
        positions."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd = self._prep(yd, self.nv, torch.float64)
        B = q.shape[0]
        p_bar, v_bar = (self._prep(_rows(t, B, 3 * self.ncp), 3 * self.ncp, torch.float64) for t in (p_bar, v_bar))
        q_bar, yd_bar = torch.empty_like(q), torch.empty_like(yd)
        _check(_lib.grbda_cuda_contact_kinematics_vjp_f64(self._h, _ptr(q), _ptr(yd), _ptr(p_bar), _ptr(v_bar),
                                                          _ptr(q_bar), _ptr(yd_bar), B, _stream()))
        return q_bar, yd_bar

    def integrate(self, q, yd, ydd, dt, out=None):
        """(q', yd', flags): semi-implicit Euler step, quaternion base by ori::integrateQuat, implicit clusters
        projected back onto phi = 0; flags[b] = 1 where that projection failed. A roll-pitch-yaw base is refused:
        flags = 1 for every state and the base positions are copied unchanged (include/grbda_cuda.h)."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd, ydd = self._prep(yd, self.nv, torch.float64), self._prep(ydd, self.nv, torch.float64)
        qo, ydo = out if out is not None else (torch.empty_like(q), torch.empty_like(yd))
        flags = torch.empty((q.shape[0],), dtype=torch.int32, device=q.device)
        _check(_lib.grbda_cuda_integrate_f64(self._h, _ptr(q), _ptr(yd), _ptr(ydd), float(dt), _ptr(qo), _ptr(ydo),
                                             _ptr(flags), q.shape[0], _stream()))
        return qo, ydo, flags

    def step(self, q, yd, tau, dt, f_ext=None, out=None):
        """One simulation step: forwardDynamics (+ external forces) and integrate."""
        import torch
        q = self._prep(q, self.nq, torch.float64)
        yd, tau = self._prep(yd, self.nv, torch.float64), self._prep(tau, self.nv, torch.float64)
        B = q.shape[0]
        if f_ext is not None:
            f_ext = self._prep(f_ext.reshape(B, -1), 6 * len(self.externalForceBodies()), torch.float64)
        qo, ydo = out if out is not None else (torch.empty_like(q), torch.empty_like(yd))
        flags = torch.empty((B,), dtype=torch.int32, device=q.device)
        _check(_lib.grbda_cuda_step_f64(self._h, _ptr(q), _ptr(yd), _ptr(tau), _ptr(f_ext), float(dt), _ptr(qo),
                                        _ptr(ydo), _ptr(flags), B, _stream()))
        return qo, ydo, flags

    def integrateVJP(self, q, yd, ydd, dt, q_out_bar, yd_out_bar):
        """(q_bar[batch, nq], yd_bar[batch, nv], ydd_bar[batch, nv], flags[batch]): the cotangents of (q', yd') =
        integrate(q, yd, ydd, dt) pulled back to the inputs; q_bar is the exact derivative of the step for every stored
        position entry, flags those of integrate (values of flagged states are meaningless; include/grbda_cuda.h)."""
        import torch
        q, q_out_bar = (self._prep(t, self.nq, torch.float64) for t in (q, q_out_bar))
        yd, ydd, yd_out_bar = (self._prep(t, self.nv, torch.float64) for t in (yd, ydd, yd_out_bar))
        q_bar, yd_bar, ydd_bar = torch.empty_like(q), torch.empty_like(yd), torch.empty_like(yd)
        flags = torch.empty((q.shape[0],), dtype=torch.int32, device=q.device)
        _check(_lib.grbda_cuda_integrate_vjp_f64(self._h, _ptr(q), _ptr(yd), _ptr(ydd), float(dt), _ptr(q_out_bar),
                                                 _ptr(yd_out_bar), _ptr(q_bar), _ptr(yd_bar), _ptr(ydd_bar), _ptr(flags),
                                                 q.shape[0], _stream()))
        return q_bar, yd_bar, ydd_bar, flags

    def stepVJP(self, q, yd, tau, dt, q_out_bar, yd_out_bar, f_ext=None):
        """(q_bar, yd_bar, tau_bar[, f_bar], flags): the cotangents of (q', yd') = step(q, yd, tau, dt, f_ext) pulled
        back to the inputs; f_bar (with f_ext only) has the shape of f_ext. The integration part of q_bar is exact, the
        dynamics part keeps the convention of forwardDynamicsVJP (include/grbda_cuda.h)."""
        import torch
        q, q_out_bar = (self._prep(t, self.nq, torch.float64) for t in (q, q_out_bar))
        yd, tau, yd_out_bar = (self._prep(t, self.nv, torch.float64) for t in (yd, tau, yd_out_bar))
        B = q.shape[0]
        f = f_bar = None
        if f_ext is not None:
            nf6 = 6 * len(self.externalForceBodies())
            f = self._prep(_rows(f_ext, B, nf6), nf6, torch.float64)
            f_bar = torch.empty_like(f)
        q_bar, yd_bar, tau_bar = torch.empty_like(q), torch.empty_like(yd), torch.empty_like(yd)
        flags = torch.empty((B,), dtype=torch.int32, device=q.device)
        _check(_lib.grbda_cuda_step_vjp_f64(self._h, _ptr(q), _ptr(yd), _ptr(tau), _ptr(f), float(dt), _ptr(q_out_bar),
                                            _ptr(yd_out_bar), _ptr(q_bar), _ptr(yd_bar), _ptr(tau_bar), _ptr(f_bar),
                                            _ptr(flags), B, _stream()))
        if f_ext is None:
            return q_bar, yd_bar, tau_bar, flags
        return q_bar, yd_bar, tau_bar, f_bar.reshape(f_ext.shape), flags

    def getMassMatrix(self, q, out=None):
        """H[batch, nv, nv]   (ClusterTreeModel::getMassMatrix)"""
        import torch
        q = self._prep(q, self.nq)
        if out is None:
            out = torch.empty((q.shape[0], self.nv, self.nv), dtype=q.dtype, device=q.device)
        fn = getattr(_lib, "grbda_cuda_mass_matrix_" + self._suffix(q))
        _check(fn(self._h, _ptr(q), _ptr(out), q.shape[0], _stream()))
        return out

    def getBiasForceVector(self, q, yd):
        """C[batch, nv] = ID(q, yd, 0)   (ClusterTreeModel::getBiasForceVector)"""
        import torch
        return self.inverseDynamics(q, yd, torch.zeros_like(yd))

    def forwardKinematics(self, q, yd, out=None):
        """(p[batch, nb, 3], R[batch, nb, 3, 3], v[batch, nb, 6]) per body: world position,
        body-to-world rotation, [world angular; world linear] velocity of the body origin.
        out: optional (p, R, v) tensors of those shapes to write into."""
        import torch
        q = self._prep(q, self.nq)
        yd = self._prep(yd, self.nv, q.dtype)
        B = q.shape[0]
        if out is not None:
            p, R, v = out
            for t, shape in ((p, (B, self.nb, 3)), (R, (B, self.nb, 3, 3)), (v, (B, self.nb, 6))):
                if tuple(t.shape) != shape or t.dtype != q.dtype or not t.is_cuda or not t.is_contiguous():
                    raise ValueError("forwardKinematics: out tensors must be contiguous CUDA tensors of shape "
                                     "(B, nb, 3), (B, nb, 3, 3), (B, nb, 6) and the dtype of q")
        else:
            p = torch.empty((B, self.nb, 3), dtype=q.dtype, device=q.device)
            R = torch.empty((B, self.nb, 3, 3), dtype=q.dtype, device=q.device)
            v = torch.empty((B, self.nb, 6), dtype=q.dtype, device=q.device)
        fn = getattr(_lib, "grbda_cuda_forward_kinematics_" + self._suffix(q))
        _check(fn(self._h, _ptr(q), _ptr(yd), _ptr(p), _ptr(R), _ptr(v), B, _stream()))
        return p, R, v

    # ---- host buffers (end-to-end path) ---------------------------------------------------------
    @staticmethod
    def _host_ptr(a, rows, cols, what):
        """Address of a float64, C-contiguous [rows, cols] host array (numpy or CPU torch tensor)."""
        if isinstance(a, np.ndarray):
            ok = a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
            ptr = a.ctypes.data
        else:
            import torch
            ok = isinstance(a, torch.Tensor) and not a.is_cuda and a.dtype == torch.float64 and a.is_contiguous()
            ptr = a.data_ptr() if ok else 0
        if not ok or tuple(a.shape) != (rows, cols):
            raise ValueError("%s: expected a float64, C-contiguous host array of shape (%d, %d)" % (what, rows, cols))
        return _vp(ptr)

    def dynamics_host(self, algo, q, yd, in3, out):
        """ID (algo=0) / FD (algo=1) on HOST arrays (numpy float64 or CPU torch tensors): H2D copy, kernel and
        D2H copy are pipelined inside the call. Page-locked arrays are used in place, pageable ones are staged."""
        B = q.shape[0]
        hp = self._host_ptr
        _check(_lib.grbda_cuda_dynamics_host_f64(self._h, algo, hp(q, B, self.nq, "q"), hp(yd, B, self.nv, "yd"),
                                                 hp(in3, B, self.nv, "in3"), hp(out, B, self.nv, "out"), B))
        return out

    def forward_inverse_host(self, q, yd, tau, ydd, tau_back):
        """One benchmark step on HOST arrays: ydd = FD(q, yd, tau), tau_back = ID(q, yd, ydd)."""
        B = q.shape[0]
        hp = self._host_ptr
        _check(_lib.grbda_cuda_forward_inverse_host_f64(self._h, hp(q, B, self.nq, "q"), hp(yd, B, self.nv, "yd"),
                                                        hp(tau, B, self.nv, "tau"), hp(ydd, B, self.nv, "ydd"),
                                                        hp(tau_back, B, self.nv, "tau_back"), B))
        return ydd, tau_back

    # ---- synthetic states / checks --------------------------------------------------------------
    def generateStates(self, count, seed=DEFAULT_SEED, first_index=0, device=None):
        """(q, yd, aux, flags): random valid states for global indices [first_index, first_index+count)."""
        import torch
        dev = torch.device("cuda", self.device if device is None else device)
        q = torch.empty((count, self.nq), dtype=torch.float64, device=dev)
        yd = torch.empty((count, self.nv), dtype=torch.float64, device=dev)
        aux = torch.empty((count, self.nv), dtype=torch.float64, device=dev)
        flags = torch.empty((count,), dtype=torch.int32, device=dev)
        _check(_lib.grbda_cuda_generate_states(self._h, seed, first_index, count, _ptr(q), _ptr(yd), _ptr(aux),
                                               _ptr(flags), _stream()))
        return q, yd, aux, flags

    def constraintViolation(self, q):
        import torch
        q = self._prep(q, self.nq, torch.float64)
        out = torch.empty((q.shape[0],), dtype=torch.float64, device=q.device)
        _check(_lib.grbda_cuda_constraint_violation_f64(self._h, _ptr(q), _ptr(out), q.shape[0], _stream()))
        return out


def checksum(x):
    """(sum, sum of absolute values) of a float64 CUDA tensor, computed on the device."""
    out = (C.c_double * 2)()
    x = x.contiguous()
    _check(_lib.grbda_cuda_checksum_f64(_ptr(x), x.numel(), out, _stream()))
    return out[0], out[1]


def __getattr__(name):
    # grbda.autograd imports torch: loaded on first use, so that importing the package does not
    if name == "autograd":
        import importlib
        return importlib.import_module(__name__ + ".autograd")
    raise AttributeError("module %r has no attribute %r" % (__name__, name))
