"""ctypes binding of the CPU oracle (oracle/libm3t_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs. The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

ROTATION_LINEAR, ROTATION_POLAR = 0, 1
EXP_RODRIGUES, EXP_PADE = 0, 1
MAX_SCHEDULE = 8

fp = C.POINTER(C.c_float)


class Intrinsics(C.Structure):
    _fields_ = [("fu", C.c_float), ("fv", C.c_float), ("ppu", C.c_float), ("ppv", C.c_float),
                ("width", C.c_int32), ("height", C.c_int32)]


class RegionParams(C.Structure):
    _fields_ = [("n_lines_max", C.c_int32), ("use_adaptive_coverage", C.c_int32),
                ("reference_contour_length", C.c_float), ("min_continuous_distance", C.c_float),
                ("function_length", C.c_int32), ("distribution_length", C.c_int32),
                ("function_amplitude", C.c_float), ("function_slope", C.c_float), ("learning_rate", C.c_float),
                ("n_global_iterations", C.c_int32), ("n_scales", C.c_int32), ("scales", C.c_int32 * MAX_SCHEDULE),
                ("n_standard_deviations", C.c_int32), ("standard_deviations", C.c_float * MAX_SCHEDULE),
                ("n_histogram_bins", C.c_int32), ("learning_rate_f", C.c_float), ("learning_rate_b", C.c_float),
                ("unconsidered_line_length", C.c_float), ("max_considered_line_length", C.c_float),
                ("measure_occlusions", C.c_int32), ("measured_depth_offset_radius", C.c_float),
                ("measured_occlusion_radius", C.c_float), ("measured_occlusion_threshold", C.c_float),
                ("n_unoccluded_iterations", C.c_int32), ("min_n_unoccluded_lines", C.c_int32),
                ("model_occlusions", C.c_int32), ("modeled_depth_offset_radius", C.c_float),
                ("modeled_occlusion_radius", C.c_float), ("modeled_occlusion_threshold", C.c_float),
                ("use_region_checking", C.c_int32)]


class DepthParams(C.Structure):
    _fields_ = [("n_points_max", C.c_int32), ("use_adaptive_coverage", C.c_int32), ("use_depth_scaling", C.c_int32),
                ("reference_surface_area", C.c_float), ("stride_length", C.c_float),
                ("n_considered_distances", C.c_int32), ("considered_distances", C.c_float * MAX_SCHEDULE),
                ("n_standard_deviations", C.c_int32), ("standard_deviations", C.c_float * MAX_SCHEDULE),
                ("measure_occlusions", C.c_int32), ("measured_depth_offset_radius", C.c_float),
                ("measured_occlusion_radius", C.c_float), ("measured_occlusion_threshold", C.c_float),
                ("n_unoccluded_iterations", C.c_int32), ("min_n_unoccluded_points", C.c_int32),
                ("model_occlusions", C.c_int32), ("modeled_depth_offset_radius", C.c_float),
                ("modeled_occlusion_radius", C.c_float), ("modeled_occlusion_threshold", C.c_float),
                ("use_silhouette_checking", C.c_int32)]


class RegionLine(C.Structure):
    _fields_ = [("model_index", C.c_int32), ("valid", C.c_int32), ("center_f_body", C.c_float * 3),
                ("center_u", C.c_float), ("center_v", C.c_float), ("normal_u", C.c_float), ("normal_v", C.c_float),
                ("delta_r", C.c_float), ("normal_component_to_scale", C.c_float), ("distribution", C.c_float * 12),
                ("mean", C.c_float), ("measured_variance", C.c_float)]


class DepthPoint(C.Structure):
    _fields_ = [("model_index", C.c_int32), ("valid", C.c_int32), ("center_f_body", C.c_float * 3),
                ("normal_f_body", C.c_float * 3), ("correspondence_center_f_camera", C.c_float * 3)]


REGION_LINE_DTYPE = np.dtype([("model_index", "<i4"), ("valid", "<i4"), ("center_f_body", "<f4", 3),
                              ("center_u", "<f4"), ("center_v", "<f4"), ("normal_u", "<f4"), ("normal_v", "<f4"),
                              ("delta_r", "<f4"), ("normal_component_to_scale", "<f4"), ("distribution", "<f4", 12),
                              ("mean", "<f4"), ("measured_variance", "<f4")])
DEPTH_POINT_DTYPE = np.dtype([("model_index", "<i4"), ("valid", "<i4"), ("center_f_body", "<f4", 3),
                              ("normal_f_body", "<f4", 3), ("correspondence_center_f_camera", "<f4", 3)])
assert REGION_LINE_DTYPE.itemsize == C.sizeof(RegionLine)
assert DEPTH_POINT_DTYPE.itemsize == C.sizeof(DepthPoint)


class Model(C.Structure):
    _fields_ = [("n_views", C.c_int32), ("n_points", C.c_int32), ("orientations", fp), ("view_scalars", fp),
                ("points", fp), ("stride_depth_offset", C.c_float), ("max_radius_depth_offset", C.c_float),
                ("max_view_scalar", C.c_float)]


class Rendering(C.Structure):
    """orc_rendering: one FocusedRenderer output (focused depth image or focused silhouette image)."""
    _fields_ = [("image", C.c_void_p), ("image_size", C.c_int32), ("pitch", C.c_size_t), ("corner_u", C.c_float),
                ("corner_v", C.c_float), ("scale", C.c_float), ("projection_term_a", C.c_float),
                ("projection_term_b", C.c_float), ("id", C.c_int32), ("visible", C.c_int32)]


class ColorFrame(C.Structure):
    _fields_ = [("intrinsics", Intrinsics), ("world2camera", C.c_float * 12), ("bgr", C.c_void_p),
                ("pitch", C.c_size_t), ("depth_rendering", C.POINTER(Rendering)),
                ("silhouette_rendering", C.POINTER(Rendering))]


class DepthFrame(C.Structure):
    _fields_ = [("intrinsics", Intrinsics), ("world2camera", C.c_float * 12), ("depth", C.c_void_p),
                ("pitch", C.c_size_t), ("depth_scale", C.c_float), ("depth_rendering", C.POINTER(Rendering)),
                ("silhouette_rendering", C.POINTER(Rendering))]


def make_rendering(r) -> Rendering:
    """r: synth.Rendering (image ndarray [size, size] u16 / u8, corner_u, corner_v, scale, a, b, id, visible)."""
    o = Rendering()
    o.image = r.image.ctypes.data
    o.image_size = r.image.shape[0]
    o.pitch = r.image.strides[0]
    o.corner_u, o.corner_v, o.scale = r.corner_u, r.corner_v, r.scale
    o.projection_term_a, o.projection_term_b = r.projection_term_a, r.projection_term_b
    o.id, o.visible = int(r.id), int(r.visible)
    return o


class Body(C.Structure):
    _fields_ = [("body2world", C.c_float * 12), ("region", C.POINTER(RegionParams)), ("region_model", C.POINTER(Model)),
                ("color", C.POINTER(ColorFrame)), ("depth", C.POINTER(DepthParams)), ("depth_model", C.POINTER(Model)),
                ("depth_frame", C.POINTER(DepthFrame)), ("histogram_f", fp), ("histogram_b", fp),
                ("tikhonov_rotation", C.c_float), ("tikhonov_translation", C.c_float), ("first_iteration", C.c_int32),
                ("lines", C.POINTER(RegionLine)), ("points", C.POINTER(DepthPoint)), ("n_lines", C.c_int32),
                ("n_points", C.c_int32), ("region_view", C.c_int32), ("depth_view", C.c_int32),
                ("region_occlusion_frame", C.POINTER(DepthFrame))]


class Link(C.Structure):
    _fields_ = [("body", C.c_int32), ("parent", C.c_int32), ("body2joint", C.c_float * 12),
                ("joint2parent", C.c_float * 12), ("free_directions", C.c_int32 * 6),
                ("fixed_body2joint_pose", C.c_int32), ("n_extra_bodies", C.c_int32), ("extra_bodies", C.c_int32 * 3)]


class Constraint(C.Structure):
    _fields_ = [("link1", C.c_int32), ("link2", C.c_int32), ("body12joint1", C.c_float * 12),
                ("body22joint2", C.c_float * 12), ("directions", C.c_int32 * 6)]


class SoftConstraint(C.Structure):
    _fields_ = [("link1", C.c_int32), ("link2", C.c_int32), ("body12joint1", C.c_float * 12),
                ("body22joint2", C.c_float * 12), ("directions", C.c_int32 * 6),
                ("max_distance_rotation", C.c_float), ("max_distance_translation", C.c_float),
                ("standard_deviation_rotation", C.c_float), ("standard_deviation_translation", C.c_float)]


class Structure(C.Structure):
    _fields_ = [("links", C.POINTER(Link)), ("n_links", C.c_int32), ("constraints", C.POINTER(Constraint)),
                ("n_constraints", C.c_int32), ("soft_constraints", C.POINTER(SoftConstraint)),
                ("n_soft_constraints", C.c_int32), ("tikhonov_rotation", C.c_float),
                ("tikhonov_translation", C.c_float)]


_libs = {}


def build():
    subprocess.run(["make", "-C", _HERE, "all"], check=True, capture_output=True)


def _load_native():
    """Compiles the -O3 -march=native build for this machine's CPU into a temporary directory (the tree may be
    read-only), loads it and removes the directory again."""
    d = tempfile.mkdtemp(prefix="m3t_oracle_native-")
    try:
        subprocess.run(["make", "-C", _HERE, "native", f"NATIVE_DIR={d}/"], check=True, capture_output=True)
        return C.CDLL(os.path.join(d, "libm3t_oracle_native.so"))
    finally:
        shutil.rmtree(d, ignore_errors=True)


def lib(native=False):
    """native=True: the -O3 -march=native build (timing only; built on the machine it runs on)."""
    key = "native" if native else "strict"
    if key in _libs:
        return _libs[key]
    if native:
        L = _load_native()
    else:
        path = os.path.join(_HERE, "libm3t_oracle.so")
        if not os.path.exists(path):
            build()
        L = C.CDLL(path)
    L.orc_region_params_default.argtypes = [C.POINTER(RegionParams)]
    L.orc_depth_params_default.argtypes = [C.POINTER(DepthParams)]
    L.orc_pose_multiply.argtypes = [fp, fp, fp]
    L.orc_pose_inverse.argtypes = [fp, fp]
    L.orc_pose_rotation.argtypes = [fp, C.c_int, fp]
    L.orc_exp_skew.argtypes = [fp, C.c_int, fp]
    L.orc_ldlt_solve.argtypes = [C.c_int, fp, fp, fp]
    L.orc_ldlt_solve.restype = C.c_int
    L.orc_function_lookup.argtypes = [C.POINTER(RegionParams), fp, fp, fp]
    L.orc_hist_clear.argtypes = [C.c_int, fp, fp]
    L.orc_hist_add.argtypes = [C.c_int, fp, C.POINTER(C.c_uint8)]
    L.orc_hist_calculate.argtypes = [C.c_int, C.c_float, fp, fp]
    L.orc_hist_get.argtypes = [C.c_int, fp, fp, C.POINTER(C.c_uint8), fp, fp]
    L.orc_closest_view.argtypes = [C.POINTER(Model), fp, C.c_int]
    L.orc_closest_view.restype = C.c_int
    L.orc_region_add_line_pixels.argtypes = [C.POINTER(RegionParams), C.POINTER(Model), C.POINTER(ColorFrame), fp,
                                             C.c_int, fp, fp]
    L.orc_region_correspondences.argtypes = [C.POINTER(RegionParams), C.POINTER(Model), C.POINTER(ColorFrame),
                                             C.POINTER(DepthFrame), fp, fp, fp, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(RegionLine), C.POINTER(C.c_int)]
    L.orc_region_correspondences.restype = C.c_int
    L.orc_region_gradient_hessian.argtypes = [C.POINTER(RegionParams), C.POINTER(ColorFrame), fp,
                                              C.POINTER(RegionLine), C.c_int, C.c_int, C.c_int, C.c_int, fp, fp]
    L.orc_depth_correspondences.argtypes = [C.POINTER(DepthParams), C.POINTER(Model), C.POINTER(DepthFrame), fp,
                                            C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(DepthPoint),
                                            C.POINTER(C.c_int)]
    L.orc_depth_correspondences.restype = C.c_int
    L.orc_depth_gradient_hessian.argtypes = [C.POINTER(DepthParams), C.POINTER(DepthFrame), fp, C.POINTER(DepthPoint),
                                             C.c_int, C.c_int, fp, fp]
    L.orc_optimize_rigid.argtypes = [fp, fp, C.c_float, C.c_float, C.c_int, fp, fp]
    L.orc_optimize_rigid.restype = C.c_int
    L.orc_start_modalities.argtypes = [C.POINTER(Body), C.c_int, C.c_int, C.c_int, C.c_int]
    L.orc_tracking_step.argtypes = [C.POINTER(Body), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_int, C.POINTER(C.c_double)]
    L.orc_calculate_results.argtypes = [C.POINTER(Body), C.c_int, C.c_int, C.c_int, C.c_int]
    L.orc_max_threads.restype = C.c_int
    sp = C.POINTER(Structure)
    L.orc_structure_dof.argtypes = [sp]
    L.orc_structure_dof.restype = C.c_int
    L.orc_structure_n_constraint_rows.argtypes = [sp]
    L.orc_structure_n_constraint_rows.restype = C.c_int
    L.orc_angle_axis.argtypes = [fp, fp, fp]
    L.orc_xcotx.argtypes = [C.c_float]
    L.orc_xcotx.restype = C.c_float
    L.orc_structure_jacobians.argtypes = [sp, C.c_int, fp]
    L.orc_constraint_residual_jacobian.argtypes = [sp, C.c_int, fp, fp, C.c_int, fp, fp]
    L.orc_constraint_residual_jacobian.restype = C.c_int
    L.orc_soft_constraint_add.argtypes = [sp, C.c_int, fp, C.c_int, fp, fp]
    L.orc_optimize_structure.argtypes = [sp, fp, fp, C.c_int, C.c_int, fp, fp]
    L.orc_optimize_structure.restype = C.c_int
    L.orc_structure_consistent_poses.argtypes = [sp, C.c_int, fp]
    L.orc_tracking_step_structures.argtypes = [C.POINTER(Body), sp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_int, C.c_int, fp, C.c_int]
    _libs[key] = L
    return L


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def ptr(a):
    return a.ctypes.data_as(fp)


def region_params(settings) -> RegionParams:
    p = RegionParams()
    lib().orc_region_params_default(C.byref(p))
    if settings is None:
        return p
    for k in ("n_lines_max", "min_continuous_distance", "function_amplitude", "function_slope", "learning_rate",
              "n_global_iterations", "n_histogram_bins", "learning_rate_f", "learning_rate_b",
              "unconsidered_line_length", "max_considered_line_length", "reference_contour_length",
              "measured_depth_offset_radius", "measured_occlusion_radius", "measured_occlusion_threshold",
              "n_unoccluded_iterations", "min_n_unoccluded_lines", "modeled_depth_offset_radius",
              "modeled_occlusion_radius", "modeled_occlusion_threshold"):
        setattr(p, k, getattr(settings, k))
    p.model_occlusions = int(settings.model_occlusions)
    p.use_region_checking = int(settings.use_region_checking)
    p.use_adaptive_coverage = int(settings.use_adaptive_coverage)
    p.measure_occlusions = int(settings.measure_occlusions)
    p.n_scales = len(settings.scales)
    p.n_standard_deviations = len(settings.standard_deviations)
    for i, s in enumerate(settings.scales):
        p.scales[i] = int(s)
    for i, s in enumerate(settings.standard_deviations):
        p.standard_deviations[i] = float(s)
    return p


def depth_params(settings) -> DepthParams:
    p = DepthParams()
    lib().orc_depth_params_default(C.byref(p))
    if settings is None:
        return p
    p.n_points_max = settings.n_points_max
    p.stride_length = settings.stride_length
    p.use_adaptive_coverage = int(settings.use_adaptive_coverage)
    p.reference_surface_area = settings.reference_surface_area
    p.use_depth_scaling = int(settings.use_depth_scaling)
    p.measure_occlusions = int(settings.measure_occlusions)
    for k in ("measured_depth_offset_radius", "measured_occlusion_radius", "measured_occlusion_threshold",
              "n_unoccluded_iterations", "min_n_unoccluded_points", "modeled_depth_offset_radius",
              "modeled_occlusion_radius", "modeled_occlusion_threshold"):
        setattr(p, k, getattr(settings, k))
    p.model_occlusions = int(settings.model_occlusions)
    p.use_silhouette_checking = int(settings.use_silhouette_checking)
    p.n_considered_distances = len(settings.considered_distances)
    p.n_standard_deviations = len(settings.standard_deviations)
    for i, s in enumerate(settings.considered_distances):
        p.considered_distances[i] = float(s)
    for i, s in enumerate(settings.standard_deviations):
        p.standard_deviations[i] = float(s)
    return p


def make_model(m) -> Model:
    """m: 3dobjecttracking_b200.synth.Model (or anything with the same attributes)."""
    om = Model()
    om.n_views, om.n_points = m.n_views, m.n_points
    om.orientations = ptr(m.orientations)
    om.view_scalars = ptr(m.view_scalars)
    om.points = ptr(m.points)
    om.stride_depth_offset = m.stride_depth_offset
    om.max_radius_depth_offset = m.max_radius_depth_offset
    om.max_view_scalar = float(m.view_scalars.max()) if m.view_scalars.size else 0.0
    return om


class OracleStructure:
    """ctypes image of one synth.StructureSpec (kept alive together with its arrays)."""

    def __init__(self, spec):
        self.spec = spec
        nl = len(spec.links)
        hard = [c for c in spec.constraints if not c.soft]
        soft = [c for c in spec.constraints if c.soft]
        self.links = (Link * nl)()
        self.constraints = (Constraint * max(1, len(hard)))()
        self.soft = (SoftConstraint * max(1, len(soft)))()
        for i, l in enumerate(spec.links):
            L_ = self.links[i]
            L_.body, L_.parent = l.body, l.parent
            L_.body2joint[:] = f32(l.body2joint).reshape(12).tolist()
            L_.joint2parent[:] = f32(l.joint2parent).reshape(12).tolist()
            L_.free_directions[:] = [int(bool(d)) for d in l.free_directions]
            L_.fixed_body2joint_pose = int(l.fixed_body2joint_pose)
            extra = tuple(getattr(l, "extra_bodies", ()) or ())
            L_.n_extra_bodies = len(extra)
            for k, e in enumerate(extra):
                L_.extra_bodies[k] = int(e)
        for arr, items in ((self.constraints, hard), (self.soft, soft)):
            for i, c in enumerate(items):
                K = arr[i]
                K.link1, K.link2 = c.link1, c.link2
                K.body12joint1[:] = f32(c.body12joint1).reshape(12).tolist()
                K.body22joint2[:] = f32(c.body22joint2).reshape(12).tolist()
                K.directions[:] = [int(bool(d)) for d in c.directions]
                if c.soft:
                    K.max_distance_rotation, K.max_distance_translation = c.max_distance_rotation, c.max_distance_translation
                    K.standard_deviation_rotation = c.standard_deviation_rotation
                    K.standard_deviation_translation = c.standard_deviation_translation
        self.n_hard, self.n_soft = len(hard), len(soft)

    def reset_joint_poses(self):
        """Link::ResetJointPoses (link.cpp:243-246)"""
        for i, l in enumerate(self.spec.links):
            self.links[i].body2joint[:] = f32(l.body2joint).reshape(12).tolist()
            self.links[i].joint2parent[:] = f32(l.joint2parent).reshape(12).tolist()

    def fill(self, S: Structure):
        S.links = C.cast(self.links, C.POINTER(Link))
        S.n_links = len(self.spec.links)
        S.constraints = C.cast(self.constraints, C.POINTER(Constraint))
        S.n_constraints = self.n_hard
        S.soft_constraints = C.cast(self.soft, C.POINTER(SoftConstraint))
        S.n_soft_constraints = self.n_soft
        S.tikhonov_rotation, S.tikhonov_translation = self.spec.tikhonov_rotation, self.spec.tikhonov_translation

    def as_struct(self) -> Structure:
        S = Structure()
        self.fill(S)
        return S

    def joint_poses(self):
        """(body2joint[n_links,3,4], joint2parent[n_links,3,4]) as they stand after the last update."""
        nl = len(self.spec.links)
        b2j = np.array([list(self.links[i].body2joint) for i in range(nl)], np.float32).reshape(nl, 3, 4)
        j2p = np.array([list(self.links[i].joint2parent) for i in range(nl)], np.float32).reshape(nl, 3, 4)
        return b2j, j2p


def _intr(i) -> Intrinsics:
    return Intrinsics(i.fu, i.fv, i.ppu, i.ppv, i.width, i.height)


class OracleTracker:
    """Drives the oracle over a synth.Workload the way Tracker drives modalities + optimizers."""

    def __init__(self, wl, rotation_mode=ROTATION_POLAR, exp_mode=EXP_PADE, n_threads=1, native=False):
        self.wl = wl
        self.L = lib(native)
        self.rotation_mode, self.exp_mode, self.n_threads = rotation_mode, exp_mode, n_threads
        nb = wl.n_bodies
        self.rp = region_params(wl.region) if wl.region else None
        self.dp = depth_params(wl.depth) if wl.depth else None
        self.rm = make_model(wl.region_model) if wl.region else None
        self.dm = make_model(wl.depth_model) if wl.depth else None
        self.bodies = (Body * nb)()
        self.color_frames = (ColorFrame * nb)()
        self.depth_frames = (DepthFrame * nb)()
        self.occlusion_frames = (DepthFrame * nb)()  # RegionModality::depth_camera_ptr (measure_occlusions)
        self.renderings = {}  # (body, key) -> Rendering, kept alive with the tracker
        rend = getattr(wl, "renderings", None) or {}

        def hook(b, key):
            r = rend.get(b, {}).get(key)
            if r is None:
                return None
            self.renderings[(b, key)] = make_rendering(r)
            return C.pointer(self.renderings[(b, key)])
        nbins = wl.region.n_histogram_bins if wl.region else 1
        self.hist_f = np.full((nb, nbins ** 3), 1.0 / nbins ** 3, np.float32)
        self.hist_b = np.full((nb, nbins ** 3), 1.0 / nbins ** 3, np.float32)
        self.lines = np.zeros((nb, max(wl.lines_per_body, 1)), REGION_LINE_DTYPE)
        self.points = np.zeros((nb, max(wl.points_per_body, 1)), DEPTH_POINT_DTYPE)
        for b in range(nb):
            B = self.bodies[b]
            if wl.region:
                cf = self.color_frames[b]
                cf.intrinsics = _intr(wl.color_intrinsics)
                cf.world2camera[:] = f32(wl.color_world2camera if getattr(wl, "color_world2camera_per_body", None) is None
                                         else wl.color_world2camera_per_body[b]).reshape(12).tolist()
                cf.bgr = wl.color_frames[b].ctypes.data
                cf.pitch = wl.color_frames[b].strides[0]
                for key, field in (("region_depth", "depth_rendering"), ("region_silhouette", "silhouette_rendering")):
                    ptr_ = hook(b, key)
                    if ptr_ is not None:
                        setattr(cf, field, ptr_)
                B.region = C.pointer(self.rp)
                B.region_model = C.pointer(self.rm)
                B.color = C.pointer(cf)
                # shared ColorHistograms (UseSharedColorHistograms): the members point at the owner's arrays
                own = b if getattr(wl, "histogram_owner", None) is None or wl.histogram_owner[b] < 0 else int(wl.histogram_owner[b])
                B.histogram_f = ptr(self.hist_f[own])
                B.histogram_b = ptr(self.hist_b[own])
                B.lines = self.lines[b].ctypes.data_as(C.POINTER(RegionLine))
                if wl.region.measure_occlusions and wl.depth_frames is not None:
                    of = self.occlusion_frames[b]
                    of.intrinsics = _intr(wl.depth_intrinsics)
                    of.world2camera[:] = f32(wl.depth_world2camera).reshape(12).tolist()
                    of.depth = wl.depth_frames[b].ctypes.data
                    of.pitch = wl.depth_frames[b].strides[0]
                    of.depth_scale = wl.depth_scale
                    B.region_occlusion_frame = C.pointer(of)
            if wl.depth:
                df = self.depth_frames[b]
                df.intrinsics = _intr(wl.depth_intrinsics)
                df.world2camera[:] = f32(wl.depth_world2camera if getattr(wl, "depth_world2camera_per_body", None) is None
                                         else wl.depth_world2camera_per_body[b]).reshape(12).tolist()
                df.depth = wl.depth_frames[b].ctypes.data
                df.pitch = wl.depth_frames[b].strides[0]
                df.depth_scale = wl.depth_scale
                for key, field in (("depth_depth", "depth_rendering"), ("depth_silhouette", "silhouette_rendering")):
                    ptr_ = hook(b, key)
                    if ptr_ is not None:
                        setattr(df, field, ptr_)
                B.depth = C.pointer(self.dp)
                B.depth_model = C.pointer(self.dm)
                B.depth_frame = C.pointer(df)
                B.points = self.points[b].ctypes.data_as(C.POINTER(DepthPoint))
            B.tikhonov_rotation = wl.tikhonov_rotation
            B.tikhonov_translation = wl.tikhonov_translation
        self.set_poses(wl.start_body2world)
        self.structures = None
        if getattr(wl, "structures", None):
            self.structure_objs = [OracleStructure(sp) for sp in wl.structures]
            self.structures = (Structure * len(self.structure_objs))()
            for i, so in enumerate(self.structure_objs):
                so.fill(self.structures[i])
            self.max_links = max(len(sp.links) for sp in wl.structures)
            self.bodyless = np.zeros((len(wl.structures), self.max_links, 12), np.float32)
            for i, sp in enumerate(wl.structures):
                for j, l in enumerate(sp.links):
                    if l.body < 0:
                        self.bodyless[i, j] = f32(l.link2world if l.link2world is not None else np.eye(4)[:3]).reshape(12)

    def set_poses(self, poses):
        p = f32(poses).reshape(self.wl.n_bodies, 12)
        for b in range(self.wl.n_bodies):
            self.bodies[b].body2world[:] = p[b].tolist()

    def reset_joint_poses(self):
        for so in (self.structure_objs if self.structures is not None else []):
            so.reset_joint_poses()

    def get_poses(self):
        return np.array([list(self.bodies[b].body2world) for b in range(self.wl.n_bodies)], np.float32).reshape(-1, 3, 4)

    def _mirror_shared_histograms(self):
        """hist_f[b] / hist_b[b] of a member of a shared object show the owner's values (the C side only writes the owner's)."""
        owner = getattr(self.wl, "histogram_owner", None)
        if owner is not None:
            for b, o in enumerate(owner):
                if o >= 0 and o != b:
                    self.hist_f[b] = self.hist_f[o]
                    self.hist_b[b] = self.hist_b[o]

    def start_modalities(self, iteration=0):
        self.L.orc_start_modalities(self.bodies, self.wl.n_bodies, iteration, self.rotation_mode, self.n_threads)
        self._mirror_shared_histograms()

    def tracking_step(self, iteration=0, n_corr=None, n_update=None, first=None, count=None, corr_begin=0):
        """Runs corr iterations [corr_begin, n_corr) for bodies [first, first+count).
        Returns the 3 phase times (s, summed over threads)."""
        n_corr = self.wl.n_corr_iterations if n_corr is None else n_corr
        n_update = self.wl.n_update_iterations if n_update is None else n_update
        first = 0 if first is None else first
        count = self.wl.n_bodies - first if count is None else count
        if self.structures is not None:  # one Optimizer per kinematic structure
            self.L.orc_tracking_step_structures(self.bodies, self.structures, len(self.structure_objs), iteration,
                                                corr_begin, n_corr, n_update, self.rotation_mode, self.exp_mode,
                                                self.n_threads, ptr(self.bodyless), self.max_links)
            return [0.0, 0.0, 0.0, 0.0]
        phases = (C.c_double * 4)()
        base = C.cast(C.byref(self.bodies, first * C.sizeof(Body)), C.POINTER(Body))
        self.L.orc_tracking_step(base, count, iteration, corr_begin, n_corr, n_update, self.rotation_mode,
                                 self.exp_mode, self.n_threads, phases)
        return list(phases)

    def calculate_results(self, iteration=0):
        self.L.orc_calculate_results(self.bodies, self.wl.n_bodies, iteration, self.rotation_mode, self.n_threads)
        self._mirror_shared_histograms()

    # fine-grained, one body
    def region_correspondences(self, b, iteration, corr):
        B = self.bodies[b]
        view = C.c_int(0)
        n = self.L.orc_region_correspondences(B.region, B.region_model, B.color, B.region_occlusion_frame, B.histogram_f, B.histogram_b,
                                              B.body2world, iteration, B.first_iteration, corr, self.rotation_mode,
                                              B.lines, C.byref(view))
        B.n_lines, B.region_view = n, view.value
        return n, view.value

    def region_gradient_hessian(self, b, corr, opt):
        B = self.bodies[b]
        g = np.zeros(6, np.float32)
        H = np.zeros(36, np.float32)
        self.L.orc_region_gradient_hessian(B.region, B.color, B.body2world, B.lines, B.n_lines, corr, opt,
                                           self.rotation_mode, ptr(g), ptr(H))
        return g, H.reshape(6, 6)

    def depth_correspondences(self, b, iteration, corr):
        B = self.bodies[b]
        view = C.c_int(0)
        n = self.L.orc_depth_correspondences(B.depth, B.depth_model, B.depth_frame, B.body2world, iteration,
                                             B.first_iteration, corr, self.rotation_mode, B.points, C.byref(view))
        B.n_points, B.depth_view = n, view.value
        return n, view.value

    def depth_gradient_hessian(self, b, corr):
        B = self.bodies[b]
        g = np.zeros(6, np.float32)
        H = np.zeros(36, np.float32)
        self.L.orc_depth_gradient_hessian(B.depth, B.depth_frame, B.body2world, B.points, B.n_points, corr, ptr(g),
                                          ptr(H))
        return g, H.reshape(6, 6)

    def optimize(self, b, g, H):
        B = self.bodies[b]
        theta = np.zeros(6, np.float32)
        g, H = f32(g), f32(H).reshape(36)
        ok = self.L.orc_optimize_rigid(ptr(g), ptr(H), B.tikhonov_rotation, B.tikhonov_translation, self.exp_mode,
                                       B.body2world, ptr(theta))
        return ok, theta
