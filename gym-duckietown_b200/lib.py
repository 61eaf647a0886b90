"""ctypes binding of libdtsim.so (include/dtsim.h).  No fallback: if the CUDA library is missing or
fails to load, importing the simulator classes raises — there is no CPU path in the product."""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional

import numpy as np

from . import assets
from .maps import KIND_ID, TILE_KINDS, MapData

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdtsim.so")

DTS_ABI_VERSION = 3
ACTION_PWM, ACTION_VEL_STEER = 0, 1
FLAG_AUTO_RESET, FLAG_DOMAIN_RAND, FLAG_DISTORTION, FLAG_DYNAMICS_RAND, FLAG_TESSELLATE = 1, 2, 4, 8, 16
IN_PROGRESS, INVALID_POSE, MAX_STEPS = 0, 1, 2
DONE_CODE_STR = {0: "in-progress", 1: "invalid-pose", 2: "max-steps-reached"}  # S:1685-1705


class DtsError(RuntimeError):
    pass


DR_INT, DR_UNIFORM, DR_NORMAL = 0, 1, 2
DR_TARGETS = {"camera_angle": 1, "camera_fov_y": 2, "camera_height": 3, "camera_noise": 4, "horz_mode": 5,
              "light_pos": 6, "trim": 7}   # DTS_DR_*; any other key is drawn and discarded (DTS_DR_NONE)
MAX_DR_OPS = 16


class DrOp(C.Structure):
    _fields_ = [("type", C.c_int32), ("size", C.c_int32), ("target", C.c_int32), ("reserved", C.c_int32),
                ("a", C.c_double * 3), ("b", C.c_double * 3)]


class Config(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_envs", C.c_int32), ("device", C.c_int32), ("cam_width", C.c_int32),
        ("cam_height", C.c_int32), ("max_steps", C.c_int32), ("frame_skip", C.c_int32), ("action_mode", C.c_int32),
        ("flags", C.c_int32), ("max_maps", C.c_int32), ("cycle_maps", C.c_int32), ("random_maps", C.c_int32),
        ("frame_rate", C.c_double), ("robot_speed", C.c_double), ("accept_start_angle_deg", C.c_double),
        ("gain", C.c_double), ("trim", C.c_double), ("radius", C.c_double), ("k", C.c_double), ("limit", C.c_double),
        ("dyn_u1", C.c_double), ("dyn_u2", C.c_double), ("dyn_u3", C.c_double), ("dyn_w1", C.c_double),
        ("dyn_w2", C.c_double), ("dyn_w3", C.c_double), ("dyn_uar", C.c_double), ("dyn_ual", C.c_double),
        ("dyn_war", C.c_double), ("dyn_wal", C.c_double), ("dyn_delay", C.c_double),
        ("seed", C.c_uint64), ("env_id_offset", C.c_int64),
        ("num_tris_distractors", C.c_int32), ("n_dr_ops", C.c_int32),
        ("color_sky", C.c_double * 3), ("color_ground", C.c_double * 3), ("dr_ops", DrOp * MAX_DR_OPS),
    ]


class Texture(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("rgba", C.c_void_p)]


class Object(C.Structure):
    _fields_ = [("pos", C.c_double * 3), ("scale", C.c_float), ("y_rot_deg", C.c_float), ("mesh_id", C.c_int32),
                ("optional", C.c_int32), ("dyn_slot", C.c_int32), ("alt_tex_from", C.c_int32), ("alt_tex_to", C.c_int32),
                ("reserved", C.c_int32)]


_DYN_SCALARS = ["safety_radius", "walk_distance", "vel", "wait_time", "wiggle", "follow_dist", "velocity", "gain",
                "trim", "radius", "k", "limit", "wheel_dist", "robot_width", "robot_length"]
DYN_FIELDS = 18   # DTS_DYN_FIELDS: px pz angle y_rot corners[8] start_x start_z wait vel time active
DYN_PX, DYN_PZ, DYN_ANGLE, DYN_YROT, DYN_CORNERS, DYN_START_X, DYN_START_Z, DYN_WAIT, DYN_VEL, DYN_TIME, DYN_ACTIVE = \
    0, 1, 2, 3, 4, 12, 13, 14, 15, 16, 17
DYN_PATTERN, DYN_SHOWN = DYN_ACTIVE, DYN_WAIT   # traffic lights (see dtsim.h)


class DynObjectC(C.Structure):
    _fields_ = [("kind", C.c_int32), ("object_index", C.c_int32), ("pos", C.c_double * 3), ("angle", C.c_double),
                ("corners", (C.c_double * 2) * 4), ("norms", (C.c_double * 2) * 2)] + \
               [(n, C.c_double) for n in _DYN_SCALARS] + [("freq", C.c_double), ("pattern", C.c_int32), ("reserved", C.c_int32)]


OBS_HWC, OBS_CHW, OBS_CWH = 0, 1, 2
OBS_U8, OBS_F32_UNIT = 0, 1
REWARD_RAW, REWARD_DT = 0, 1
ACTIONS_CONTINUOUS, ACTIONS_DISCRETE3 = 0, 1


class OutputFormat(C.Structure):
    _fields_ = [("obs_layout", C.c_int32), ("obs_dtype", C.c_int32), ("reward_mode", C.c_int32),
                ("action_map", C.c_int32), ("action_vel_scale", C.c_double)]


class Mesh(C.Structure):
    _fields_ = [("tri_offset", C.c_int32), ("tri_count", C.c_int32), ("seg_flat_tex", C.c_int32), ("reserved", C.c_int32)]


RENDER_SEGMENT, RENDER_TOP_DOWN = 1, 2


class MapBlob(C.Structure):
    _fields_ = [
        ("tile_size", C.c_double), ("grid_w", C.c_int32), ("grid_h", C.c_int32),
        ("tile_kind", C.c_void_p), ("tile_angle", C.c_void_p), ("tile_drivable", C.c_void_p), ("tile_tex", C.c_void_p),
        ("tile_curve_off", C.c_void_p), ("tile_curve_cnt", C.c_void_p), ("n_curves", C.c_int32), ("curves", C.c_void_p),
        ("n_coll", C.c_int32), ("coll_corners", C.c_void_p), ("coll_norms", C.c_void_p), ("coll_centers", C.c_void_p),
        ("coll_radii", C.c_void_p), ("n_objects", C.c_int32), ("objects", C.c_void_p), ("n_meshes", C.c_int32),
        ("meshes", C.c_void_p), ("n_tris", C.c_int32), ("tri_pos", C.c_void_p), ("tri_nrm", C.c_void_p),
        ("tri_uv", C.c_void_p), ("tri_col", C.c_void_p), ("tri_tex", C.c_void_p), ("n_textures", C.c_int32),
        ("textures", C.c_void_p), ("start_tile", C.c_int32 * 2), ("n_dyn", C.c_int32), ("has_start_pose", C.c_int32),
        ("dyn", C.c_void_p), ("start_pose", C.c_double * 3),
        ("tex_segment", C.c_void_p), ("agent_mesh", C.c_int32), ("reserved2", C.c_int32),
    ]


_EP_FIELDS = ["map_id", "pos_x", "pos_z", "angle", "wheel_dist", "trim", "cam_height", "cam_angle_deg",
              "cam_fov_y_deg", "cam_noise", "horizon_color", "light_ambient", "light_diffuse", "light_pos",
              "light_stale", "ground_color", "obj_hidden"]
_EP_DTYPES = {"map_id": np.int32, "pos_x": np.float64, "pos_z": np.float64, "angle": np.float64,
              "wheel_dist": np.float64, "trim": np.float64, "cam_height": np.float32, "cam_angle_deg": np.float32,
              "cam_fov_y_deg": np.float32, "cam_noise": np.float32, "horizon_color": np.float32,
              "light_ambient": np.float32, "light_diffuse": np.float32, "light_pos": np.float32,
              "light_stale": np.int32, "ground_color": np.float32, "obj_hidden": np.uint32}
_EP_WIDTH = {"cam_noise": 3, "horizon_color": 3, "light_ambient": 3, "light_diffuse": 3, "light_pos": 4,
             "ground_color": 3, "obj_hidden": 8}


class EpisodeParams(C.Structure):
    _fields_ = [(f, C.c_void_p) for f in _EP_FIELDS]


_STATE_FIELDS = [("pos_x", np.float64), ("pos_z", np.float64), ("angle", np.float64), ("speed", np.float64),
                 ("reward", np.float64), ("lane_dist", np.float64), ("lane_dot", np.float64),
                 ("lane_angle_rad", np.float64), ("prox_penalty", np.float64), ("wheel_dist", np.float64),
                 ("step_count", np.int32), ("tile_i", np.int32), ("tile_j", np.int32), ("map_id", np.int32),
                 ("episode", np.int32), ("done_code", np.uint8), ("in_lane", np.uint8), ("collided", np.uint8)]


class StateView(C.Structure):
    _fields_ = [(n, C.c_void_p) for n, _ in _STATE_FIELDS]


_lib = None


def load() -> C.CDLL:
    """Load libdtsim.so; (re)build it first when it is missing or older than csrc/ or dtsim.h and nvcc is on PATH
    (build.build checks the mtimes).  Fails loudly: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    import shutil
    from . import build as _b
    if os.environ.get("DTS_NO_REBUILD"):     # load the library as built (e.g. a -DDTS_STATS build), never rebuild it
        pass
    elif shutil.which("nvcc"):
        _b.build(force=False)
    elif not os.path.exists(LIB_PATH):
        raise DtsError(f"{LIB_PATH} is missing and nvcc is not available to build it")
    elif _b.needs_build():
        import warnings
        warnings.warn("libdtsim.so is older than its sources and nvcc is not available: loading the stale library")
    try:
        lib = C.CDLL(LIB_PATH)
    except OSError as e:  # no fallback, by design
        raise DtsError(f"cannot load {LIB_PATH}: {e}") from e
    vp, i = C.c_void_p, C.c_int
    lib.dts_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    lib.dts_upload_map.argtypes = [vp, i, C.POINTER(MapBlob)]
    lib.dts_set_fisheye_lut.argtypes = [vp, vp, vp, i, i]
    lib.dts_reset.argtypes = [vp, vp, C.POINTER(EpisodeParams), vp]
    lib.dts_reset_random.argtypes = [vp, vp, vp]
    lib.dts_seed_streams.argtypes = [vp, vp, vp]
    lib.dts_step.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.dts_render.argtypes = [vp, vp, vp]
    lib.dts_get_state.argtypes = [vp, C.POINTER(StateView)]
    lib.dts_query_poses.argtypes = [vp, i, i, i, vp, vp, vp, vp, vp]
    lib.dts_assign_maps.argtypes = [vp, vp, vp, vp]
    lib.dts_set_resize.argtypes = [vp, i, i]
    lib.dts_set_render_mode.argtypes = [vp, i]
    lib.dts_resize_frames.argtypes = [vp, vp, vp, vp]
    lib.dts_blend4.argtypes = [vp, vp, vp, vp, C.c_uint64, vp]
    lib.dts_set_timing.argtypes = [vp, C.c_double, i, i]
    lib.dts_status.argtypes = [vp]
    lib.dts_profile_enable.argtypes = [vp, i]
    lib.dts_profile_read.argtypes = [vp, vp, vp]
    lib.dts_set_output_format.argtypes = [vp, C.POINTER(OutputFormat)]
    lib.dts_get_dyn_state.argtypes = [vp, i, C.POINTER(vp), C.POINTER(C.c_int32)]
    lib.dts_gather_alloc.argtypes = [vp, C.c_uint64, i, i, vp, C.POINTER(vp)]
    lib.dts_gather_open.argtypes = [vp, vp]
    lib.dts_gather_next.argtypes = [vp]
    lib.dts_comm_load.argtypes = [vp, C.c_char_p]
    lib.dts_comm_unique_id.argtypes = [vp, vp]
    lib.dts_comm_init.argtypes = [vp, vp, i, i]
    lib.dts_allgather_obs.argtypes = [vp, vp, vp, C.c_uint64, vp]
    lib.dts_launch_count.argtypes = [vp]
    lib.dts_debug_counters.argtypes = [vp, vp]
    lib.dts_debug_episode.argtypes = [vp, i, vp]
    lib.dts_debug_frame.argtypes = [vp, i, vp, vp, vp, vp, i]
    lib.dts_launch_count.restype = C.c_uint64
    lib.dts_last_error.argtypes = [vp]
    lib.dts_last_error.restype = C.c_char_p
    lib.dts_destroy.argtypes = [vp]
    lib.dts_destroy.restype = None
    _lib = lib
    return lib


EXPORTS = ["dts_create", "dts_upload_map", "dts_set_fisheye_lut", "dts_reset", "dts_seed_streams", "dts_reset_random", "dts_step",
           "dts_render", "dts_get_state", "dts_query_poses", "dts_assign_maps", "dts_set_resize", "dts_set_render_mode", "dts_resize_frames", "dts_blend4", "dts_set_timing", "dts_status", "dts_profile_enable", "dts_profile_read", "dts_get_dyn_state", "dts_set_output_format", "dts_gather_alloc", "dts_gather_open", "dts_gather_next", "dts_comm_load", "dts_comm_unique_id", "dts_comm_init",
           "dts_allgather_obs", "dts_launch_count", "dts_debug_counters", "dts_debug_episode", "dts_debug_frame", "dts_last_error", "dts_destroy"]


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class MapBlobHolder:
    """Flattens a MapData (tiles, curves, OBBs, placed meshes, textures) into a dts_map_blob and keeps
    the numpy buffers alive for the duration of the upload."""

    def __init__(self, md: MapData, user_tile_start=None):
        k = self.keep = {}
        k["kind"] = np.ascontiguousarray(md.tile_kind, np.int8)
        k["angle"] = np.ascontiguousarray(md.tile_angle, np.int8)
        k["drv"] = np.ascontiguousarray(md.tile_drivable, np.uint8)
        # textures: one per tile kind present, then the mesh textures
        tex_imgs: List[np.ndarray] = []
        kind_tex = {}
        for kid in sorted(set(int(x) for x in md.tile_kind if x >= 0)):
            kind_tex[kid] = len(tex_imgs)
            tex_imgs.append(np.ascontiguousarray(assets.tile_texture(TILE_KINDS[kid])))
        n_tile_tex = len(tex_imgs)
        k["tex"] = np.array([kind_tex.get(int(x), -1) for x in md.tile_kind], np.int16)
        k["coff"] = np.ascontiguousarray(md.tile_curve_off, np.int32)
        k["ccnt"] = np.ascontiguousarray(md.tile_curve_cnt, np.int32)
        k["curves"] = np.ascontiguousarray(md.curves, np.float64)
        k["cc"] = np.ascontiguousarray(md.coll_corners, np.float64)
        k["cn"] = np.ascontiguousarray(md.coll_norms, np.float64)
        k["ce"] = np.ascontiguousarray(md.coll_centers, np.float64)
        k["cr"] = np.ascontiguousarray(md.coll_radii, np.float64)
        mesh_list = list(md.meshes)
        agent_mesh = len(mesh_list)                       # self.mesh = get_duckiebot_mesh("red") S:864: top-down views draw it
        mesh_list.append(assets.get_mesh("duckiebot"))
        meshes = (Mesh * max(1, len(mesh_list)))()
        pos, nrm, uv, col, ttex = [], [], [], [], []
        off = 0
        alt_of_mesh = {}
        mesh_tex_range = []
        for mi, m in enumerate(mesh_list):
            base = len(tex_imgs)
            tex_imgs.extend(np.ascontiguousarray(t) for t in m.textures)
            for slot, img in getattr(m, "alt_textures", {}).items():   # traffic-light card for pattern 1
                alt_of_mesh[mi] = (base + slot, len(tex_imgs))
                tex_imgs.append(np.ascontiguousarray(img))
            mesh_tex_range.append((base, len(tex_imgs)))
            meshes[mi] = Mesh(off, len(m.tri_pos), -1, 0)
            off += len(m.tri_pos)
            pos.append(m.tri_pos); nrm.append(m.tri_nrm); uv.append(m.tri_uv); col.append(m.tri_col)
            ttex.append(np.where(m.tri_tex >= 0, m.tri_tex + base, -1).astype(np.int16))
        # segment=True assets: tiles keep their lane markings or go black (graphics.py:70-130); every chunk of a mesh
        # shows the flat class colour gen_segmentation_color(mesh_name) (objmesh.py:260-290)
        seg_of = np.arange(len(tex_imgs), dtype=np.int64)
        n_plain = len(tex_imgs)
        for kid, ti in kind_tex.items():
            seg_of[ti] = len(tex_imgs)
            tex_imgs.append(np.ascontiguousarray(assets.segment_tile_texture(TILE_KINDS[kid], tex_imgs[ti])))
        for mi, m in enumerate(mesh_list):
            name = "sign_generic" if m.name.startswith("sign") else m.name
            meshes[mi].seg_flat_tex = len(tex_imgs)
            seg_of[mesh_tex_range[mi][0]:mesh_tex_range[mi][1]] = len(tex_imgs)
            tex_imgs.append(assets.flat_texture(assets.gen_segmentation_color(name)))
        seg_full = np.arange(len(tex_imgs), dtype=np.int16)
        seg_full[:n_plain] = seg_of
        k["seg"] = seg_full
        cat = lambda lst, shape, dt: (np.ascontiguousarray(np.concatenate(lst, 0), dt) if lst else np.zeros(shape, dt))
        k["tpos"] = cat(pos, (0, 3, 3), np.float32); k["tnrm"] = cat(nrm, (0, 3, 3), np.float32)
        k["tuv"] = cat(uv, (0, 3, 2), np.float32); k["tcol"] = cat(col, (0, 3, 3), np.float32)
        k["ttex"] = cat(ttex, (0,), np.int16)
        objs = (Object * max(1, len(md.objects)))()
        slot_of = {d.object_index: s for s, d in enumerate(md.dyn_objects)}
        for oi, o in enumerate(md.objects):
            objs[oi] = Object((C.c_double * 3)(*[float(v) for v in o.pos]), float(o.scale),
                              float(np.rad2deg(o.angle)), o.mesh_id, int(o.optional), slot_of.get(oi, -1),
                              *(alt_of_mesh.get(o.mesh_id, (-1, -1)) if o.kind == "trafficlight" else (-1, -1)), 0)  # y_rot O:57
        dyn = (DynObjectC * max(1, len(md.dyn_objects)))()
        for s, d in enumerate(md.dyn_objects):
            c = dyn[s]
            c.kind, c.object_index, c.angle = int(d.kind), int(d.object_index), float(d.angle)
            for i in range(3):
                c.pos[i] = float(d.pos[i])
            for i in range(4):
                c.corners[i][0], c.corners[i][1] = float(d.corners[i][0]), float(d.corners[i][1])
            for i in range(2):
                c.norms[i][0], c.norms[i][1] = float(d.axes[i][0]), float(d.axes[i][1])
            for n in _DYN_SCALARS:
                setattr(c, n, float(getattr(d, n)))
            c.freq, c.pattern = float(d.freq), int(d.pattern)
        k["dyn"] = dyn
        texs = (Texture * max(1, len(tex_imgs)))()
        for ti, im in enumerate(tex_imgs):
            texs[ti] = Texture(im.shape[1], im.shape[0], im.ctypes.data)
        k["tex_imgs"], k["meshes"], k["objs"], k["texs"] = tex_imgs, meshes, objs, texs
        self.blob = MapBlob(
            md.tile_size, md.grid_w, md.grid_h, _ptr(k["kind"]), _ptr(k["angle"]), _ptr(k["drv"]), _ptr(k["tex"]),
            _ptr(k["coff"]), _ptr(k["ccnt"]), len(md.curves), _ptr(k["curves"]), md.n_coll, _ptr(k["cc"]),
            _ptr(k["cn"]), _ptr(k["ce"]), _ptr(k["cr"]), len(md.objects), C.cast(objs, C.c_void_p), len(mesh_list),
            C.cast(meshes, C.c_void_p), off, _ptr(k["tpos"]), _ptr(k["tnrm"]), _ptr(k["tuv"]), _ptr(k["tcol"]),
            _ptr(k["ttex"]), len(tex_imgs), C.cast(texs, C.c_void_p),
            (C.c_int32 * 2)(*(user_tile_start if user_tile_start else
                              (md.start_tile if md.start_tile is not None else (-1, -1)))),   # S:659-671
            len(md.dyn_objects), int(md.start_pose is not None), C.cast(dyn, C.c_void_p),
            (C.c_double * 3)(*((float(md.start_pose[0][0]), float(md.start_pose[0][2]), float(md.start_pose[1]))
                               if md.start_pose is not None else (0.0, 0.0, 0.0))),
            _ptr(k["seg"]), agent_mesh, 0)
        self.agent_mesh, self.n_tile_tex = agent_mesh, n_tile_tex


class _CudaArray:
    """Minimal __cuda_array_interface__ wrapper so torch can view library-owned device memory."""

    def __init__(self, ptr: int, n: int, dtype):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": np.dtype(dtype).str, "data": (ptr, False),
                                         "version": 2}


class Sim:
    """Thin OO veneer over the C handle; every method maps 1:1 to an entry point of dtsim.h."""

    def __init__(self, cfg: Config):
        self.lib = load()
        self.h = C.c_void_p()
        self.cfg = cfg
        if self.lib.dts_create(C.byref(cfg), C.byref(self.h)):
            raise DtsError("dts_create: " + self.lib.dts_last_error(None).decode())

    def _check(self, rc: int, what: str):
        if rc:
            raise DtsError(f"{what}: {self.lib.dts_last_error(self.h).decode()}")

    def upload_map(self, map_id: int, md: MapData, user_tile_start=None):
        holder = MapBlobHolder(md, user_tile_start)
        self._check(self.lib.dts_upload_map(self.h, map_id, C.byref(holder.blob)), "dts_upload_map")

    def set_fisheye_lut(self, rmapx: np.ndarray, rmapy: np.ndarray):
        rx, ry = np.ascontiguousarray(rmapx, np.float32), np.ascontiguousarray(rmapy, np.float32)
        self._check(self.lib.dts_set_fisheye_lut(self.h, _ptr(rx), _ptr(ry), rx.shape[1], rx.shape[0]),
                    "dts_set_fisheye_lut")

    def reset(self, mask_ptr: Optional[int], params: dict, stream: int = 0):
        n = self.cfg.num_envs
        keep, ep = [], EpisodeParams()
        for f in _EP_FIELDS:
            v = params.get(f)
            if v is None:
                continue
            a = np.ascontiguousarray(v, _EP_DTYPES[f])
            want = (n, _EP_WIDTH[f]) if f in _EP_WIDTH else (n,)
            if a.shape != want:
                raise ValueError(f"episode param {f}: shape {a.shape}, expected {want}")
            keep.append(a)
            setattr(ep, f, a.ctypes.data)
        self._check(self.lib.dts_reset(self.h, mask_ptr, C.byref(ep), stream), "dts_reset")

    def seed_streams(self, generators, mask: Optional[np.ndarray] = None):
        """Upload one numpy PCG64 stream per env (list of numpy.random.Generator) for device-side resets."""
        n = self.cfg.num_envs
        arr = np.zeros((n, 6), np.uint64)
        m64 = (1 << 64) - 1
        for e, g in enumerate(generators):
            st = g.bit_generator.state
            if st["bit_generator"] != "PCG64":
                raise ValueError("device streams are PCG64")
            s, inc = st["state"]["state"], st["state"]["inc"]
            arr[e] = (s >> 64, s & m64, inc >> 64, inc & m64, st["has_uint32"], st["uinteger"])
        mk = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        self._check(self.lib.dts_seed_streams(self.h, _ptr(mk), _ptr(arr)), "dts_seed_streams")

    def reset_random(self, mask_ptr: Optional[int], stream: int = 0):
        self._check(self.lib.dts_reset_random(self.h, mask_ptr, stream), "dts_reset_random")

    def step(self, actions_ptr: int, obs_ptr: Optional[int], reward_ptr: int, done_ptr: int, stream: int = 0):
        self._check(self.lib.dts_step(self.h, actions_ptr, obs_ptr, reward_ptr, done_ptr, stream), "dts_step")

    def render(self, obs_ptr: int, stream: int = 0):
        self._check(self.lib.dts_render(self.h, obs_ptr, stream), "dts_render")

    def set_output_format(self, obs_layout=OBS_HWC, obs_dtype=OBS_U8, reward_mode=REWARD_RAW,
                          action_map=ACTIONS_CONTINUOUS, action_vel_scale=1.0):
        f = OutputFormat(obs_layout, obs_dtype, reward_mode, action_map, float(action_vel_scale))
        self._check(self.lib.dts_set_output_format(self.h, C.byref(f)), "dts_set_output_format")

    def state_arrays(self) -> dict:
        v = StateView()
        self._check(self.lib.dts_get_state(self.h, C.byref(v)), "dts_get_state")
        return {n: _CudaArray(getattr(v, n), self.cfg.num_envs, dt) for n, dt in _STATE_FIELDS}

    def query_poses(self, map_id: int, x, z, angle, safety=1.0, hidden=None, dyn_env: int = -1, stream: int = 0):
        """dyn_env: the env whose dynamic obstacles the predicates see (-1: static scene only).  Runs on `stream`,
        i.e. after the steps already queued there, and returns when the answers are on the host."""
        q = np.empty((len(x), 4), np.float64)
        q[:, 0], q[:, 1], q[:, 2], q[:, 3] = x, z, angle, safety
        outd = np.empty((len(x), 4), np.float64)
        outi = np.empty((len(x), 8), np.int32)
        hid = None if hidden is None else np.ascontiguousarray(hidden, np.uint32)
        self._check(self.lib.dts_query_poses(self.h, map_id, int(dyn_env), len(x), _ptr(q), _ptr(hid), _ptr(outd), _ptr(outi),
                                             stream), "dts_query_poses")
        return outd, outi

    def assign_maps(self, mask_ptr: Optional[int], map_ids: np.ndarray, stream: int = 0):
        """randomize_maps_on_reset (host-drawn): new map ids + re-created obstacles, nothing else (dts_assign_maps)."""
        ids = np.ascontiguousarray(map_ids, np.int32)
        if ids.shape != (self.cfg.num_envs,):
            raise ValueError("map_ids must have one entry per env")
        self._check(self.lib.dts_assign_maps(self.h, mask_ptr, _ptr(ids), stream), "dts_assign_maps")

    def set_render_mode(self, segment: bool = False, top_down: bool = False):
        self._check(self.lib.dts_set_render_mode(self.h, (RENDER_SEGMENT if segment else 0) | (RENDER_TOP_DOWN if top_down else 0)),
                    "dts_set_render_mode")

    def set_resize(self, out_w: int, out_h: int):
        self._check(self.lib.dts_set_resize(self.h, int(out_w), int(out_h)), "dts_set_resize")

    def resize_frames(self, src_ptr: int, dst_ptr: int, stream: int = 0):
        self._check(self.lib.dts_resize_frames(self.h, src_ptr, dst_ptr, stream), "dts_resize_frames")

    def blend4(self, frame_ptrs, weights, out_ptr: int, n: int, stream: int = 0):
        fp = (C.c_void_p * 4)(*frame_ptrs)
        w = (C.c_double * 4)(*[float(x) for x in weights])
        self._check(self.lib.dts_blend4(self.h, fp, w, out_ptr, n, stream), "dts_blend4")

    def set_timing(self, delta_time: float, frame_skip: int, action_mode: int):
        self._check(self.lib.dts_set_timing(self.h, float(delta_time), int(frame_skip), int(action_mode)), "dts_set_timing")

    def status(self) -> int:
        """Sticky status bits, read without synchronising (bit 0: a frame overflowed its render frame memory)."""
        return int(self.lib.dts_status(self.h))

    def profile(self, level):
        """0 / False off; 1 / True: CUDA events around k_raster only; 2: around every render kernel."""
        self._check(self.lib.dts_profile_enable(self.h, int(level)), "dts_profile_enable")

    def profile_read(self):
        """(dict kernel -> summed ms, frames) since the last read; synchronises."""
        ms = np.zeros(8, np.float64)
        fr = C.c_int64()
        self._check(self.lib.dts_profile_read(self.h, _ptr(ms), C.byref(fr)), "dts_profile_read")
        names = ["k_frame_setup", "k_geometry", "k_bin", "k_raster", "post"]
        return {n: float(ms[k]) for k, n in enumerate(names)}, int(fr.value)

    def dyn_state(self, map_id: int = 0):
        """(device array f64[DYN_FIELDS * n_dyn * num_envs], n_dyn) of map `map_id`'s dynamic obstacles, or (None, 0)."""
        p, nd = C.c_void_p(), C.c_int32()
        self._check(self.lib.dts_get_dyn_state(self.h, map_id, C.byref(p), C.byref(nd)), "dts_get_dyn_state")
        if not nd.value:
            return None, 0
        return _CudaArray(p.value, DYN_FIELDS * nd.value * self.cfg.num_envs, np.float64), nd.value

    def launch_count(self) -> int:
        return int(self.lib.dts_launch_count(self.h))

    def debug_episode(self, env: int) -> dict:
        raw = np.zeros(36, np.float32)
        self._check(self.lib.dts_debug_episode(self.h, env, _ptr(raw)), "dts_debug_episode")
        return dict(cam_height=raw[0], cam_angle_deg=raw[1], cam_fov_y_deg=raw[2], cam_noise=raw[4:7], horizon=raw[8:11],
                    ambient=raw[12:15], diffuse=raw[16:19], light_eye=raw[20:24], ground=raw[24:27],
                    hidden=raw[28:36].view(np.uint32))

    def debug_frame(self, env: int, n_cells: int) -> dict:
        """Frame setup of `env` in the last render: V f64[12], P f32[4], counts, lattice f32[n_cells, 64, 3] (NaN = culled)."""
        V, P, cnt = np.zeros(12), np.zeros(4, np.float32), np.zeros(4, np.int32)
        lat = np.zeros((n_cells, 64, 3), np.float32)
        self._check(self.lib.dts_debug_frame(self.h, env, _ptr(V), _ptr(P), _ptr(cnt), _ptr(lat), n_cells), "dts_debug_frame")
        return dict(V=V, P=P, n_prims=int(cnt[0]), n_lat=int(cnt[1]), overflow=int(cnt[2]), batch_pairs=int(cnt[3]), lattice=lat)

    def debug_counters(self) -> np.ndarray:
        out = np.zeros(32, np.int32)
        self._check(self.lib.dts_debug_counters(self.h, _ptr(out)), "dts_debug_counters")
        return out

    def close(self):
        if self.h:
            self.lib.dts_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def default_config(**kw) -> Config:
    """Reference defaults: Simulator.__init__ (S:207-232), DuckietownEnv.__init__ (E:15), DB18 nominal."""
    c = Config(
        abi_version=DTS_ABI_VERSION, num_envs=1, device=0, cam_width=640, cam_height=480, max_steps=1500, frame_skip=1,
        action_mode=ACTION_VEL_STEER, flags=0, max_maps=1, cycle_maps=0, random_maps=0, frame_rate=30.0, robot_speed=1.2,
        accept_start_angle_deg=60.0, gain=1.0, trim=0.0, radius=0.0318, k=27.0, limit=1.0,
        dyn_u1=5.0, dyn_u2=0.0, dyn_u3=0.0, dyn_w1=4.0, dyn_w2=0.0, dyn_w3=0.0, dyn_uar=1.5, dyn_ual=1.5,
        dyn_war=15.0, dyn_wal=15.0, dyn_delay=0.15, seed=0, env_id_offset=0, num_tris_distractors=12, n_dr_ops=0)
    c.color_sky[:] = (0.45, 0.82, 1.0)      # BLUE_SKY S:108
    c.color_ground[:] = (0.15, 0.15, 0.15)  # S:228
    for k_, v in kw.items():
        if not hasattr(c, k_):
            raise TypeError(f"unknown config field {k_}")
        if k_ in ("color_sky", "color_ground"):
            getattr(c, k_)[:] = [float(x) for x in v]
        elif k_ == "dr_ops":
            set_dr_ops(c, v)
        else:
            setattr(c, k_, v)
    return c


def dr_ops_from_config(cfg: dict) -> list:
    """Randomizer table (randomization/randomizer.py:19-89) -> list of (type, size, target, a[3], b[3]) in the
    reference's draw order (sorted keys).  `cfg` is the parsed JSON: {key: {"type": "int" | "uniform" | "normal", ...}}."""
    ops = []
    for key in sorted(cfg):
        d = cfg[key]
        t = d["type"]
        size = d.get("size", 1)
        if t == "int":
            ty, a, b = DR_INT, d["low"], d["high"]
        elif t == "uniform":
            ty, a, b = DR_UNIFORM, d["low"], d["high"]
        elif t == "normal":
            ty, a, b = DR_NORMAL, d["loc"], d["scale"]
        else:
            raise NotImplementedError("You've specified an unsupported distribution type")   # randomizer.py:79
        a3 = np.broadcast_to(np.asarray(a, np.float64), (min(int(size), 3),) if np.ndim(a) == 0 else np.shape(a))
        b3 = np.broadcast_to(np.asarray(b, np.float64), (min(int(size), 3),) if np.ndim(b) == 0 else np.shape(b))
        if int(size) > 3 and (np.ndim(a) or np.ndim(b)):
            raise ValueError(f"DR key {key}: array bounds with size > 3 are not supported")
        av, bv = np.zeros(3), np.zeros(3)
        av[:len(a3)], bv[:len(b3)] = a3, b3
        ops.append((ty, int(size), DR_TARGETS.get(key, 0), av, bv))
    if len(ops) > MAX_DR_OPS:
        raise ValueError(f"at most {MAX_DR_OPS} randomization keys")
    return ops


def set_dr_ops(c: Config, ops: list):
    c.n_dr_ops = len(ops)
    for k, (ty, size, target, a, b) in enumerate(ops):
        c.dr_ops[k].type, c.dr_ops[k].size, c.dr_ops[k].target = ty, size, target
        c.dr_ops[k].a[:] = [float(x) for x in a]
        c.dr_ops[k].b[:] = [float(x) for x in b]
