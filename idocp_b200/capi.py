"""ctypes binding of the C-ABI (include/idocp_b200.h).

The product library is the nvcc-built ``idocp_b200/libidocp_b200.so`` (sm_100a).  There is no CPU
fallback: if the library is missing, or no CUDA device is usable, loading / creation raises.
``Library(path)`` with an explicit path exists so that the CPU-only test-suite can load the SIMT
emulator build of the same sources (tests/emu) -- it is never chosen automatically.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# IDOCP_B200_LIBRARY: another nvcc build of the same sources (A/B variants from tools/build_variant.py); never a fallback
DEFAULT_LIBRARY = os.environ.get("IDOCP_B200_LIBRARY") or os.path.join(_HERE, "libidocp_b200.so")

DIMV = 7
NUM_CONSTRAINTS = 6
DC_DOUBLES = 323   # IDOCP_B200_DC_DOUBLES (include/idocp_b200.h)
ROBOT_IIWA14 = 0
SOLVER_UNOCP = 0
SOLVER_UNPARNMPC = 1

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class Problem(C.Structure):
    """idocp_b200_problem (include/idocp_b200.h)."""
    _fields_ = [
        ("robot", C.c_int), ("N", C.c_int), ("T", C.c_double),
        ("q_ref", C.c_double * DIMV), ("v_ref", C.c_double * DIMV), ("u_ref", C.c_double * DIMV),
        ("q_weight", C.c_double * DIMV), ("v_weight", C.c_double * DIMV), ("a_weight", C.c_double * DIMV),
        ("u_weight", C.c_double * DIMV), ("qf_weight", C.c_double * DIMV), ("vf_weight", C.c_double * DIMV),
        ("q_min", C.c_double * DIMV), ("q_max", C.c_double * DIMV),
        ("v_max", C.c_double * DIMV), ("u_max", C.c_double * DIMV),
        ("barrier", C.c_double), ("fraction_rate", C.c_double),
        ("task_enabled", C.c_int),
        ("task_q_weight", C.c_double * 6), ("task_qf_weight", C.c_double * 6),
        ("task_center", C.c_double * 3), ("task_radius", C.c_double),
        ("task_t0", C.c_double), ("task_tf", C.c_double),
        ("task_rot_ref", C.c_double * 9),
        ("enable_acceleration_limit", C.c_int * 2), ("a_min", C.c_double * DIMV), ("a_max", C.c_double * DIMV),
    ]


MAX_GRID = 1024
MAX_EVENTS = 64


class ScheduledStage(C.Structure):
    """idocp_b200_scheduled_stage."""
    _fields_ = [("kind", C.c_int), ("index", C.c_int), ("t", C.c_double), ("dt", C.c_double),
                ("contact_phase", C.c_int), ("constraint_stage", C.c_int), ("before_impulse", C.c_int),
                ("switching_impulse", C.c_int)]


class OCPDiscretization(C.Structure):
    """idocp_b200_ocp_discretization."""
    _fields_ = [
        ("well_defined", C.c_int), ("N", C.c_int), ("N_impulse", C.c_int), ("N_lift", C.c_int),
        ("t", C.c_double * (MAX_GRID + 1)), ("dt", C.c_double * (MAX_GRID + 1)),
        ("contact_phase", C.c_int * (MAX_GRID + 1)),
        ("impulse_index_after_time_stage", C.c_int * (MAX_GRID + 1)),
        ("lift_index_after_time_stage", C.c_int * (MAX_GRID + 1)),
        ("time_stage_before_impulse", C.c_int * MAX_EVENTS), ("time_stage_before_lift", C.c_int * MAX_EVENTS),
        ("t_impulse", C.c_double * MAX_EVENTS), ("t_lift", C.c_double * MAX_EVENTS),
        ("dt_aux", C.c_double * MAX_EVENTS), ("dt_lift", C.c_double * MAX_EVENTS),
        ("num_stages", C.c_int),
        ("stages", ScheduledStage * (MAX_GRID + 1 + 3 * MAX_EVENTS)),
    ]


FB_NUM_CONSTRAINTS = 8


class FbProblem(C.Structure):
    """idocp_b200_fb_problem (include/idocp_b200.h): OCPSolver problem data of the floating-base robot."""
    _fields_ = [
        ("T", C.c_double), ("N", C.c_int), ("max_num_impulse", C.c_int),
        ("q_weight", C.c_double * 18), ("v_weight", C.c_double * 18), ("a_weight", C.c_double * 18),
        ("qf_weight", C.c_double * 18), ("vf_weight", C.c_double * 18), ("qi_weight", C.c_double * 18),
        ("vi_weight", C.c_double * 18), ("dvi_weight", C.c_double * 18),
        ("f_weight", C.c_double * 12), ("f_ref", C.c_double * 12), ("fi_weight", C.c_double * 12), ("fi_ref", C.c_double * 12),
        ("q_min", C.c_double * 12), ("q_max", C.c_double * 12), ("v_max", C.c_double * 12), ("u_max", C.c_double * 12),
        ("mu", C.c_double), ("barrier", C.c_double), ("fraction_rate", C.c_double),
        ("enable", C.c_int * FB_NUM_CONSTRAINTS),
        ("cone_nonlinear", C.c_int * 2), ("enable_acceleration_limit", C.c_int * 2),
        ("a_min", C.c_double * 12), ("a_max", C.c_double * 12),
        ("enable_contact_distance", C.c_int),
    ]


class Idocp_b200Error(RuntimeError):
    pass


EXPORTS = [
    "idocp_b200_problem_default", "idocp_b200_create", "idocp_b200_destroy", "idocp_b200_set_solution",
    "idocp_b200_init_constraints", "idocp_b200_init_backward_correction", "idocp_b200_update_solution",
    "idocp_b200_update_solution_device", "idocp_b200_compute_kkt_residual",
    "idocp_b200_compute_kkt_residual_device", "idocp_b200_kkt_error", "idocp_b200_get_solution", "idocp_b200_get_stage_solution",
    "idocp_b200_get_direction", "idocp_b200_get_constraint_data", "idocp_b200_get_step_sizes",
    "idocp_b200_get_unkkt", "idocp_b200_check_cost_derivatives", "idocp_b200_get_status", "idocp_b200_is_feasible",
    "idocp_b200_clear_line_search_filter", "idocp_b200_sync", "idocp_b200_launch_count", "idocp_b200_stream",
    "idocp_b200_set_task_reference", "idocp_b200_set_profiling", "idocp_b200_get_profile", "idocp_b200_set_pipelining",
    "idocp_b200_contact_sequence_create", "idocp_b200_contact_sequence_destroy",
    "idocp_b200_contact_sequence_set_uniform", "idocp_b200_contact_sequence_push_back",
    "idocp_b200_contact_sequence_pop_back", "idocp_b200_contact_sequence_pop_front",
    "idocp_b200_contact_sequence_update_event_time", "idocp_b200_contact_sequence_set_contact_points",
    "idocp_b200_contact_sequence_counts", "idocp_b200_contact_sequence_get_phase",
    "idocp_b200_contact_sequence_get_impulse", "idocp_b200_contact_sequence_get_lift_time",
    "idocp_b200_discretize_ocp", "idocp_b200_last_error", "idocp_b200_version",
    "idocp_b200_fb_create", "idocp_b200_fb_destroy", "idocp_b200_fb_set_solution", "idocp_b200_fb_set_cost_reference",
    "idocp_b200_fb_discretize", "idocp_b200_fb_init_constraints", "idocp_b200_fb_update_solution",
    "idocp_b200_fb_compute_kkt_residual", "idocp_b200_fb_kkt_error", "idocp_b200_fb_get_step_sizes", "idocp_b200_fb_get",
    "idocp_b200_fb_sync", "idocp_b200_fb_launch_count", "idocp_b200_fb_stream", "idocp_b200_fb_set_profiling",
    "idocp_b200_fb_get_profile", "idocp_b200_fb_record_bytes", "idocp_b200_fb_problem_default",
    "idocp_b200_fb_total_weight", "idocp_b200_fb_contact_frame_positions", "idocp_b200_fb_clear_line_search_filter",
    "idocp_b200_fb_set_strict_discretization",
    "idocp_b200_fb_create_sharded", "idocp_b200_fb_sharded_destroy", "idocp_b200_fb_sharded_num_shards", "idocp_b200_fb_sharded_shard",
    "idocp_b200_fb_sharded_set_solution", "idocp_b200_fb_sharded_set_cost_reference", "idocp_b200_fb_sharded_discretize",
    "idocp_b200_fb_sharded_init_constraints", "idocp_b200_fb_sharded_set_strict_discretization",
    "idocp_b200_fb_sharded_update_solution", "idocp_b200_fb_sharded_compute_kkt_residual", "idocp_b200_fb_sharded_kkt_error",
    "idocp_b200_fb_sharded_clear_line_search_filter", "idocp_b200_fb_sharded_get_step_sizes", "idocp_b200_fb_sharded_get",
    "idocp_b200_fb_sharded_sync", "idocp_b200_fb_sharded_launch_count",
    "idocp_b200_create_sharded", "idocp_b200_sharded_destroy", "idocp_b200_sharded_num_shards", "idocp_b200_sharded_shard",
    "idocp_b200_sharded_set_solution", "idocp_b200_sharded_init_constraints", "idocp_b200_sharded_init_backward_correction",
    "idocp_b200_sharded_set_task_reference", "idocp_b200_sharded_update_solution", "idocp_b200_sharded_compute_kkt_residual",
    "idocp_b200_sharded_kkt_error", "idocp_b200_sharded_get_solution", "idocp_b200_sharded_get_stage_solution",
    "idocp_b200_sharded_get_step_sizes", "idocp_b200_sharded_get_status", "idocp_b200_sharded_clear_line_search_filter",
    "idocp_b200_sharded_sync",
]


class Library:
    def __init__(self, path=None):
        path = path or DEFAULT_LIBRARY
        if not os.path.exists(path):
            raise Idocp_b200Error(
                "CUDA extension %s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)" % path)
        self.path = path
        L = C.CDLL(path)
        for name in EXPORTS:
            if not hasattr(L, name):
                raise Idocp_b200Error("library %s does not export %s" % (path, name))
        L.idocp_b200_last_error.restype = C.c_char_p
        L.idocp_b200_version.restype = C.c_char_p
        L.idocp_b200_update_solution.argtypes = [C.c_void_p, C.c_double, _dp, _dp, C.c_int]
        L.idocp_b200_update_solution_device.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_int]
        L.idocp_b200_compute_kkt_residual.argtypes = [C.c_void_p, C.c_double, _dp, _dp]
        L.idocp_b200_compute_kkt_residual_device.argtypes = [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]
        L.idocp_b200_init_backward_correction.argtypes = [C.c_void_p, C.c_double]
        L.idocp_b200_create.argtypes = [C.POINTER(Problem), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.idocp_b200_destroy.argtypes = [C.c_void_p]
        L.idocp_b200_set_solution.argtypes = [C.c_void_p, C.c_char_p, _dp, C.c_int]
        L.idocp_b200_init_constraints.argtypes = [C.c_void_p]
        L.idocp_b200_kkt_error.argtypes = [C.c_void_p, _dp]
        L.idocp_b200_get_solution.argtypes = [C.c_void_p, C.c_char_p, _dp]
        L.idocp_b200_get_stage_solution.argtypes = [C.c_void_p, C.c_char_p, C.c_int, _dp]
        L.idocp_b200_get_direction.argtypes = [C.c_void_p, C.c_char_p, _dp]
        L.idocp_b200_get_constraint_data.argtypes = [C.c_void_p, C.c_char_p, _dp]
        L.idocp_b200_get_step_sizes.argtypes = [C.c_void_p, _dp, _dp]
        L.idocp_b200_get_unkkt.argtypes = [C.c_void_p, C.c_int, _dp, _dp]
        L.idocp_b200_check_cost_derivatives.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, C.c_double, _dp]
        L.idocp_b200_get_status.argtypes = [C.c_void_p, _ip]
        L.idocp_b200_is_feasible.argtypes = [C.c_void_p, _ip]
        L.idocp_b200_clear_line_search_filter.argtypes = [C.c_void_p]
        L.idocp_b200_sync.argtypes = [C.c_void_p]
        L.idocp_b200_set_task_reference.argtypes = [C.c_void_p, _dp]
        L.idocp_b200_contact_sequence_create.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.idocp_b200_contact_sequence_destroy.argtypes = [C.c_void_p]
        L.idocp_b200_contact_sequence_set_uniform.argtypes = [C.c_void_p, _ip, _dp]
        L.idocp_b200_contact_sequence_push_back.argtypes = [C.c_void_p, _ip, _dp, C.c_double]
        L.idocp_b200_contact_sequence_pop_back.argtypes = [C.c_void_p]
        L.idocp_b200_contact_sequence_pop_front.argtypes = [C.c_void_p]
        L.idocp_b200_contact_sequence_update_event_time.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double]
        L.idocp_b200_contact_sequence_set_contact_points.argtypes = [C.c_void_p, C.c_int, _dp]
        L.idocp_b200_contact_sequence_counts.argtypes = [C.c_void_p, _ip, _ip, _ip]
        L.idocp_b200_contact_sequence_get_phase.argtypes = [C.c_void_p, C.c_int, _ip, _dp]
        L.idocp_b200_contact_sequence_get_impulse.argtypes = [C.c_void_p, C.c_int, _ip, _dp, _dp]
        L.idocp_b200_contact_sequence_get_lift_time.argtypes = [C.c_void_p, C.c_int, _dp]
        L.idocp_b200_discretize_ocp.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_double,
                                                C.POINTER(OCPDiscretization)]
        L.idocp_b200_launch_count.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
        L.idocp_b200_stream.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.idocp_b200_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.idocp_b200_set_pipelining.argtypes = [C.c_void_p, C.c_int]
        L.idocp_b200_get_profile.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), _dp,
                                             C.POINTER(C.c_longlong)]
        L.idocp_b200_fb_create.argtypes = [C.POINTER(FbProblem), C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.idocp_b200_fb_destroy.argtypes = [C.c_void_p]
        L.idocp_b200_fb_set_solution.argtypes = [C.c_void_p, C.c_char_p, _dp, C.c_int]
        L.idocp_b200_fb_set_cost_reference.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, _dp]
        L.idocp_b200_fb_discretize.argtypes = [C.c_void_p, C.c_double, C.c_int, _ip, _ip, _dp, _dp, _ip, _ip, _ip]
        L.idocp_b200_fb_init_constraints.argtypes = [C.c_void_p, C.c_double]
        L.idocp_b200_fb_update_solution.argtypes = [C.c_void_p, C.c_double, _dp, _dp, C.c_int]
        L.idocp_b200_fb_compute_kkt_residual.argtypes = [C.c_void_p, C.c_double, _dp, _dp]
        L.idocp_b200_fb_kkt_error.argtypes = [C.c_void_p, _dp]
        L.idocp_b200_fb_get_step_sizes.argtypes = [C.c_void_p, _dp]
        L.idocp_b200_fb_get.argtypes = [C.c_void_p, C.c_int, C.c_char_p, _dp]
        L.idocp_b200_fb_sync.argtypes = [C.c_void_p]
        L.idocp_b200_fb_clear_line_search_filter.argtypes = [C.c_void_p]
        L.idocp_b200_fb_set_strict_discretization.argtypes = [C.c_void_p, C.c_int]
        L.idocp_b200_fb_launch_count.argtypes = [C.c_void_p, C.POINTER(C.c_longlong)]
        L.idocp_b200_fb_stream.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.idocp_b200_fb_set_profiling.argtypes = [C.c_void_p, C.c_int]
        L.idocp_b200_fb_get_profile.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), _dp, C.POINTER(C.c_longlong)]
        # the sharded twins take the same arguments behind the handle
        for name in ("set_solution", "set_cost_reference", "discretize", "init_constraints", "update_solution", "compute_kkt_residual",
                     "kkt_error", "get_step_sizes", "get", "sync", "clear_line_search_filter", "set_strict_discretization",
                     "launch_count"):
            getattr(L, "idocp_b200_fb_sharded_" + name).argtypes = getattr(L, "idocp_b200_fb_" + name).argtypes
        L.idocp_b200_fb_create_sharded.argtypes = [C.POINTER(FbProblem), C.c_void_p, C.c_int, _ip, C.c_int, C.POINTER(C.c_void_p)]
        L.idocp_b200_fb_problem_default.argtypes = [C.POINTER(FbProblem)]
        L.idocp_b200_fb_total_weight.restype = C.c_double
        L.idocp_b200_fb_contact_frame_positions.argtypes = [_dp, _dp]
        L.idocp_b200_create_sharded.argtypes = [C.POINTER(Problem), C.c_int, C.c_int, _ip, C.c_int, C.POINTER(C.c_void_p)]
        for name in ("set_solution", "init_constraints", "init_backward_correction", "set_task_reference", "update_solution",
                     "compute_kkt_residual", "kkt_error", "get_solution", "get_stage_solution", "get_step_sizes", "get_status",
                     "clear_line_search_filter", "sync"):
            getattr(L, "idocp_b200_sharded_" + name).argtypes = getattr(L, "idocp_b200_" + name).argtypes
        for family in ("", "fb_"):
            getattr(L, "idocp_b200_%ssharded_destroy" % family).argtypes = [C.c_void_p]
            getattr(L, "idocp_b200_%ssharded_num_shards" % family).argtypes = [C.c_void_p, _ip, _ip]
            getattr(L, "idocp_b200_%ssharded_shard" % family).argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]
        self.L = L

    def check(self, rc):
        if rc < 0:
            raise Idocp_b200Error("idocp_b200 error %d: %s" % (rc, self.L.idocp_b200_last_error().decode()))
        return rc

    def entry(self, family, name, sharded):
        """The entry point idocp_b200_<family><name> of a solver handle, or its sharded twin idocp_b200_<family>sharded_<name>
        (same arguments); raises for an entry point that has no sharded twin."""
        full = "idocp_b200_%s%s%s" % (family, "sharded_" if sharded else "", name)
        try:
            return getattr(self.L, full)
        except AttributeError:
            raise Idocp_b200Error("%s does not exist: a sharded solver has one single-device solver per device" % full) from None

    def version(self):
        return self.L.idocp_b200_version().decode()

    def default_problem(self, robot=ROBOT_IIWA14):
        p = Problem()
        self.check(self.L.idocp_b200_problem_default(robot, C.byref(p)))
        return p


_default = None


def default_library():
    """The CUDA library; raises when it has not been built."""
    global _default
    if _default is None:
        _default = Library()
    return _default


def dptr(a):
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_dp)
