"""ctypes binding of include/cuda_trace.h (libcuda_trace.so) -- the reference-facing boundary.

There is no fallback of any kind: if the CUDA library is missing, or no B200 is present,
``CudaTrace()`` raises.
"""
import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libcuda_trace.so")

MISS = 0xFFFFFFFF
VARIANT_MT = 0
VARIANT_BARY = 1
QUERY_CLOSEST = 0
QUERY_OCCLUSION = 1
FLAG_GAMMA = 1
FLAG_KEEP_HITS = 2
FLAG_ORTHO = 4              # camera.h:25-36; the frame's fov_xs then carries the width of the viewing volume
FLAG_SHADE_FACE_NORMAL = 8  # renderer.cpp:116
FLAG_SHADE_DEPTH = 16       # renderer.cpp:118

_F32P = C.POINTER(C.c_float)
_U32P = C.POINTER(C.c_uint32)
_U64P = C.POINTER(C.c_uint64)


class Frame(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("spp", C.c_uint32), ("variant", C.c_uint32),
                ("flags", C.c_uint32), ("fov_xs", C.c_float), ("aspect", C.c_float), ("cam_mat", C.c_float * 16)]


class TileRect(C.Structure):
    _fields_ = [("x0", C.c_uint32), ("y0", C.c_uint32), ("x1", C.c_uint32), ("y1", C.c_uint32)]


class GridDesc(C.Structure):
    _fields_ = [("dim", C.c_uint32 * 3), ("aabb_min", C.c_float * 3), ("aabb_max", C.c_float * 3),
                ("cell_wdh", C.c_float), ("inv_cell_wdh", C.c_float), ("num_cells", C.c_uint64),
                ("num_refs", C.c_uint64)]


class RayBatch(C.Structure):
    """cuda_trace_ray_batch: every pointer is device memory"""
    _fields_ = [("n", C.c_uint32), ("kind", C.c_uint32), ("variant", C.c_uint32), ("t_max_all", C.c_float),
                ("origins", C.c_void_p), ("dirs", C.c_void_p), ("t_max", C.c_void_p), ("tri_idx", C.c_void_p),
                ("t", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p), ("occluded", C.c_void_p)]


class CountersC(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("cells", C.c_uint64), ("tri_tests", C.c_uint64), ("hits", C.c_uint64)]


# every symbol include/cuda_trace.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "cuda_trace_init": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "cuda_trace_init_devices": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    "cuda_trace_destroy": (None, [C.c_void_p]),
    "cuda_trace_last_error": (C.c_char_p, [C.c_void_p]),
    "cuda_trace_device_count": (C.c_int, []),
    "cuda_trace_set_shard": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "cuda_trace_set_shard_signals": (C.c_int, [C.c_void_p, C.c_int]),
    "cuda_trace_upload_scene": (C.c_int, [C.c_void_p, _F32P, C.c_uint32, _U32P, C.c_uint32, C.c_uint32]),
    "cuda_trace_suggest_grid_res": (C.c_uint32, [C.c_uint32]),
    "cuda_trace_upload_scene_with_grid": (C.c_int, [C.c_void_p, _F32P, C.c_uint32, _U32P, C.c_uint32,
                                                    C.POINTER(GridDesc), _U64P, _U32P]),
    "cuda_trace_download_grid": (C.c_int, [C.c_void_p, C.POINTER(GridDesc), _U64P, _U32P]),
    "cuda_trace_download_distance_map": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]),
    "cuda_trace_download_screen_boxes": (C.c_int, [C.c_void_p, _F32P, C.c_uint64, C.POINTER(C.c_uint64),
                                                   C.POINTER(C.c_uint32), C.POINTER(C.c_int)]),
    "cuda_trace_tiles": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.POINTER(TileRect), C.c_uint32, _U32P]),
    "cuda_trace_tiles_into": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.POINTER(TileRect), C.c_uint32, C.POINTER(_U32P),
                                        C.c_void_p, C.c_void_p]),
    "cuda_trace_tiles_async": (C.c_int, [C.c_void_p, C.POINTER(Frame), C.POINTER(TileRect), C.c_uint32]),
    "cuda_trace_sync": (C.c_int, [C.c_void_p]),
    "cuda_trace_read_framebuffer": (C.c_int, [C.c_void_p, _U32P]),
    "cuda_trace_cancel": (C.c_int, [C.c_void_p]),
    "cuda_trace_last_kernel_ms": (C.c_int, [C.c_void_p, _F32P]),
    "cuda_trace_download_hits": (C.c_int, [C.c_void_p, _U32P, _F32P, _F32P, _F32P]),
    "cuda_trace_intersect_rays": (C.c_int, [C.c_void_p, C.c_uint32, _F32P, _F32P, C.c_uint32, _U32P, _F32P,
                                            _F32P, _F32P]),
    "cuda_trace_mailbox_stats": (C.c_int, [C.c_void_p, _U64P, _U64P]),
    "cuda_trace_query_rays": (C.c_int, [C.c_void_p, C.POINTER(RayBatch), C.c_void_p]),
    "cuda_trace_intersect_rays_brute_force": (C.c_int, [C.c_void_p, C.c_uint32, _F32P, _F32P, _U32P, _F32P, _F32P, _F32P]),
    "cuda_trace_band_shares": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                         _U32P, _U32P, _U32P, _U32P, _U32P]),
    "cuda_trace_last_call_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "cuda_trace_download_strip_cycles": (C.c_int, [C.c_void_p, _U32P, C.c_uint64, C.POINTER(C.c_uint64)]),
    "cuda_trace_ray_march": (C.c_int, [C.c_void_p, C.c_uint32, _F32P, _F32P, _U32P, _F32P]),
    "cuda_trace_sample_table": (C.c_int, [C.c_void_p, C.c_uint32, _F32P]),
    "cuda_trace_qmc_sequence": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _U32P, C.c_uint32, C.c_uint32, C.c_uint32,
                                          C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_double)]),
    "cuda_trace_qmc_cranley_patterson": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.c_double, C.c_uint32,
                                                   C.POINTER(C.c_double)]),
    "cuda_trace_set_counting": (C.c_int, [C.c_void_p, C.c_int]),
    "cuda_trace_get_counters": (C.c_int, [C.c_void_p, C.POINTER(CountersC)]),
    "cuda_trace_host_alloc": (C.c_void_p, [C.c_size_t]),
    "cuda_trace_host_free": (None, [C.c_void_p]),
    "cuda_trace_kernel_launches": (C.c_uint64, [C.c_void_p]),
    "cuda_trace_prepare_framebuffer": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "cuda_trace_export_framebuffer": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cuda_trace_import_framebuffer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    "cuda_trace_framebuffer_device_ptr": (C.c_void_p, [C.c_void_p]),
    "cuda_trace_stream": (C.c_void_p, [C.c_void_p]),
}

_lib = None


def load_library():
    """dlopen libcuda_trace.so and bind every declared symbol.  Raises if the library is absent:
    the product path has no other implementation to fall back to."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(LIB_PATH + " is missing: build it with "
                               "`python cpp-11-ray-trace-march-framework_b200/build.py` "
                               "(there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class CudaTraceError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("cuda_trace error %d: %s" % (code, msg))
        self.code = code


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


def full_frame_tiles(width, height, tiles_x=12, tiles_y=9):
    """The reference's fixed 12 x 9 tile layout (framebuffer.h:87-88, framebuffer.cpp:106-117):
    tile size = floor(size / count), the last column / row absorbs the remainder."""
    tw, th = width // tiles_x, height // tiles_y
    out = []
    for y in range(tiles_y):
        for x in range(tiles_x):
            out.append((x * tw, y * th, width if x == tiles_x - 1 else (x + 1) * tw,
                        height if y == tiles_y - 1 else (y + 1) * th))
    return out


def band_shares(width, height, spp, rects, world, chunk=32):
    """Host arithmetic of the overlapped read-back (no device needed): -> dict(shares [world, 32], gpus_in_band [32],
    band_rows, n_bands, pieces_per_strip) for the frame layout ``rects``."""
    lib = load_library()
    tiles, n_tiles = CudaTrace.make_tiles(rects)
    shares, gpus = np.zeros((world, 32), np.uint32), np.zeros(32, np.uint32)
    rows, nb, pieces = C.c_uint32(), C.c_uint32(), C.c_uint32()
    rc = lib.cuda_trace_band_shares(width, height, spp, tiles, n_tiles, world, chunk, _p(shares, _U32P), _p(gpus, _U32P),
                                    C.byref(rows), C.byref(nb), C.byref(pieces))
    if rc:
        raise ValueError("cuda_trace_band_shares: bad arguments")
    return dict(shares=shares, gpus_in_band=gpus, band_rows=rows.value, n_bands=nb.value, pieces_per_strip=pieces.value)


MEASURE_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libcuda_trace_measure.so")
_measure_lib = None


def load_measure_library():
    """dlopen libcuda_trace_measure.so (include/cuda_trace_measure.h): roofline ceilings, L2 flush, arithmetic
    self-check.  Measurement code -- the product library does not link it."""
    global _measure_lib
    if _measure_lib is None:
        if not os.path.exists(MEASURE_LIB_PATH):
            raise RuntimeError(MEASURE_LIB_PATH + " is missing: build it with "
                               "`python cpp-11-ray-trace-march-framework_b200/build.py`")
        lib = C.CDLL(MEASURE_LIB_PATH)
        lib.rtm_measure_peaks.restype = C.c_int
        lib.rtm_measure_peaks.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        lib.rtm_measure_flush_l2.restype = C.c_int
        lib.rtm_measure_flush_l2.argtypes = [C.c_int]
        lib.rtm_measure_check_fast_arith.restype = C.c_int
        lib.rtm_measure_check_fast_arith.argtypes = [C.c_int, C.c_uint64, C.c_uint32, C.c_int, C.c_int,
                                                     C.POINTER(C.c_ulonglong)]
        _measure_lib = lib
    return _measure_lib


def measure_peaks(device=0):
    """-> (FP32 non-FMA T instr-flop/s, L2 read GB/s) measured on ``device`` (csrc/measure.cu)."""
    lib = load_measure_library()
    a, b = C.c_double(), C.c_double()
    rc = lib.rtm_measure_peaks(device, C.byref(a), C.byref(b))
    if rc:
        raise RuntimeError("rtm_measure_peaks failed: %d" % rc)
    return a.value, b.value


def flush_l2(device=0):
    """Evict the L2 of ``device`` (between timed frames; synchronises the device)."""
    rc = load_measure_library().rtm_measure_flush_l2(device)
    if rc:
        raise RuntimeError("rtm_measure_flush_l2 failed: %d" % rc)


def check_fast_arith(n, seed=1, exp_lo=-40, exp_hi=40, device=0):
    """-> (rcp, div, sqrt) mismatch counts of the range-check-free sequences against the IEEE intrinsics."""
    bad = (C.c_ulonglong * 3)()
    rc = load_measure_library().rtm_measure_check_fast_arith(device, n, seed, exp_lo, exp_hi, bad)
    if rc:
        raise RuntimeError("rtm_measure_check_fast_arith failed: %d" % rc)
    return tuple(int(x) for x in bad)


class PinnedImage:
    """[H, W] uint32 numpy view of page-locked host memory (cuda_trace_host_alloc)."""

    def __init__(self, width, height):
        self.lib = load_library()
        self.ptr = self.lib.cuda_trace_host_alloc(width * height * 4)
        if not self.ptr:
            raise MemoryError("cuda_trace_host_alloc failed")
        buf = (C.c_uint32 * (width * height)).from_address(self.ptr)
        self.array = np.frombuffer(buf, np.uint32).reshape(height, width)

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            self.lib.cuda_trace_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        self.close()


class CudaTrace:
    """One cuda_trace_ctx.  ``n_gpus`` devices (0..n-1) or an explicit ``devices`` list."""

    def __init__(self, n_gpus=1, devices=None):
        self.lib = load_library()
        self.h = C.c_void_p()
        self.devices = list(devices) if devices is not None else list(range(n_gpus))
        if devices is not None:
            arr = (C.c_int * len(devices))(*devices)
            rc = self.lib.cuda_trace_init_devices(arr, len(devices), C.byref(self.h))
        else:
            rc = self.lib.cuda_trace_init(n_gpus, C.byref(self.h))
        if rc:
            msg = self.lib.cuda_trace_last_error(None).decode()
            self.h = None
            raise CudaTraceError(rc, msg)
        self._pinned = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.cuda_trace_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def _ck(self, rc):
        if rc:
            raise CudaTraceError(rc, self.lib.cuda_trace_last_error(self.h).decode())

    # -- scene
    def upload_scene(self, vtx, tri, grid_res=64):
        vtx = np.ascontiguousarray(vtx, np.float32)
        tri = np.ascontiguousarray(tri, np.uint32)
        self._ck(self.lib.cuda_trace_upload_scene(self.h, _p(vtx, _F32P), len(vtx), _p(tri, _U32P), len(tri), grid_res))

    def upload_scene_with_grid(self, vtx, tri, grid):
        vtx = np.ascontiguousarray(vtx, np.float32)
        tri = np.ascontiguousarray(tri, np.uint32)
        d = GridDesc()
        for k in range(3):
            d.dim[k] = int(grid["dim"][k])
            d.aabb_min[k] = float(grid["aabb_min"][k])
            d.aabb_max[k] = float(grid["aabb_max"][k])
        d.cell_wdh = float(grid["cell_wdh"])
        d.inv_cell_wdh = float(grid["inv_cell_wdh"])
        off = np.ascontiguousarray(grid["cell_offset"], np.uint64)
        idx = np.ascontiguousarray(grid["tri_index"], np.uint32)
        d.num_cells = len(off) - 1
        d.num_refs = len(idx)
        self._ck(self.lib.cuda_trace_upload_scene_with_grid(self.h, _p(vtx, _F32P), len(vtx), _p(tri, _U32P),
                                                            len(tri), C.byref(d), _p(off, _U64P),
                                                            _p(idx, _U32P) if len(idx) else None))

    def download_grid(self):
        d = GridDesc()
        self._ck(self.lib.cuda_trace_download_grid(self.h, C.byref(d), None, None))
        off = np.zeros(d.num_cells + 1, np.uint64)
        idx = np.zeros(max(int(d.num_refs), 1), np.uint32)
        self._ck(self.lib.cuda_trace_download_grid(self.h, C.byref(d), _p(off, _U64P), _p(idx, _U32P)))
        return dict(dim=np.array(list(d.dim), np.uint32), aabb_min=np.array(list(d.aabb_min), np.float32),
                    aabb_max=np.array(list(d.aabb_max), np.float32), cell_wdh=np.float32(d.cell_wdh),
                    inv_cell_wdh=np.float32(d.inv_cell_wdh), cell_offset=off, tri_index=idx[:int(d.num_refs)])

    def download_distance_map(self):
        """-> uint8 array [dim_y + 2, dim_z + 2, dim_x + 2] of the padded grid, or None when the scene has none"""
        n = C.c_uint64(0)
        self._ck(self.lib.cuda_trace_download_distance_map(self.h, None, C.byref(n)))
        if n.value == 0:
            return None
        out = np.zeros(n.value, np.uint8)
        self._ck(self.lib.cuda_trace_download_distance_map(self.h, out.ctypes.data_as(C.c_void_p), C.byref(n)))
        d = GridDesc()
        self._ck(self.lib.cuda_trace_download_grid(self.h, C.byref(d), None, None))
        return out.reshape(d.dim[1] + 2, d.dim[2] + 2, d.dim[0] + 2)

    def download_screen_boxes(self):
        """-> (boxes float32 [num_pairs, 4] {xmin, xmax, ymin, ymax}, small, cull_on): the screen boxes of device 0
        for the camera of the last frame that built them; num_pairs = 0 when none are built"""
        n, small, on = C.c_uint64(0), C.c_uint32(0), C.c_int(0)
        self._ck(self.lib.cuda_trace_download_screen_boxes(self.h, None, 0, C.byref(n), C.byref(small), C.byref(on)))
        out = np.zeros((n.value, 4), np.float32)
        if n.value:
            self._ck(self.lib.cuda_trace_download_screen_boxes(self.h, _p(out, _F32P), out.size, C.byref(n),
                                                               C.byref(small), C.byref(on)))
        return out, int(small.value), bool(on.value)

    # -- frames
    @staticmethod
    def make_frame(width, height, spp, cam16, fov_xs, aspect, variant=VARIANT_MT, gamma=True, keep_hits=False,
                   ortho_width=None, shade_mode=0):
        """ortho_width: orthographic camera of that width (replaces fov_xs); shade_mode 1 / 2: face normal / depth"""
        f = Frame()
        f.width, f.height, f.spp, f.variant = width, height, spp, variant
        f.flags = ((FLAG_GAMMA if gamma else 0) | (FLAG_KEEP_HITS if keep_hits else 0) |
                   (FLAG_ORTHO if ortho_width is not None else 0) |
                   (FLAG_SHADE_FACE_NORMAL if shade_mode == 1 else 0) | (FLAG_SHADE_DEPTH if shade_mode == 2 else 0))
        f.fov_xs, f.aspect = float(fov_xs if ortho_width is None else ortho_width), float(aspect)
        cam16 = np.asarray(cam16, np.float32).reshape(16)
        for i in range(16):
            f.cam_mat[i] = float(cam16[i])
        return f

    @staticmethod
    def make_tiles(rects):
        """list of (x0, y0, x1, y1) -> (TileRect array, count); a result of make_tiles passes through, so a
        caller rendering the same layout every frame converts it once."""
        if isinstance(rects, tuple) and len(rects) == 2 and isinstance(rects[0], C.Array):
            return rects
        arr = (TileRect * max(len(rects), 1))()
        for i, r in enumerate(rects):
            arr[i].x0, arr[i].y0, arr[i].x1, arr[i].y1 = [int(v) for v in r]
        return arr, len(rects)

    def trace_tiles(self, frame, rects=None, out=None, want_image=True):
        """Render ``rects`` (default: the reference's 12x9 layout of the whole frame) and return
        the host image [H, W] uint32 (row 0 = y 0)."""
        if rects is None:
            rects = full_frame_tiles(frame.width, frame.height)
        tiles, n_tiles = self.make_tiles(rects)
        if want_image and out is None:
            out = np.zeros((frame.height, frame.width), np.uint32)
        self._ck(self.lib.cuda_trace_tiles(self.h, C.byref(frame), tiles, n_tiles,
                                           _p(out, _U32P) if want_image else None))
        return out

    def trace_tiles_into(self, frame, rects=None):
        """cuda_trace_tiles_into: every tile into its own page-locked buffer.  -> (list of [th, tw] uint32 arrays,
        list of tile-index groups in the order the library reported them complete)"""
        if rects is None:
            rects = full_frame_tiles(frame.width, frame.height)
        tiles, n_tiles = self.make_tiles(rects)
        pinned = [PinnedImage(max(tiles[i].x1 - tiles[i].x0, 1), max(tiles[i].y1 - tiles[i].y0, 1)) for i in range(n_tiles)]
        ptrs = (_U32P * max(n_tiles, 1))(*[C.cast(p.ptr, _U32P) for p in pinned])
        groups = []
        cb_type = C.CFUNCTYPE(None, _U32P, C.c_uint32, C.c_void_p)
        cb = cb_type(lambda idx, n, user: groups.append([int(idx[k]) for k in range(n)]))
        rc = self.lib.cuda_trace_tiles_into(self.h, C.byref(frame), tiles, n_tiles, ptrs, C.cast(cb, C.c_void_p), None)
        out = [p.array.copy() for p in pinned]
        for p in pinned:
            p.close()
        self._ck(rc)
        return out, groups

    def trace_tiles_async(self, frame, rects=None):
        if rects is None:
            rects = full_frame_tiles(frame.width, frame.height)
        tiles, n_tiles = self.make_tiles(rects)
        self._ck(self.lib.cuda_trace_tiles_async(self.h, C.byref(frame), tiles, n_tiles))

    def sync(self):
        self._ck(self.lib.cuda_trace_sync(self.h))

    def read_framebuffer(self, out):
        self._ck(self.lib.cuda_trace_read_framebuffer(self.h, _p(out, _U32P)))
        return out

    def cancel(self):
        self._ck(self.lib.cuda_trace_cancel(self.h))

    def last_kernel_ms(self):
        ms = C.c_float()
        self._ck(self.lib.cuda_trace_last_kernel_ms(self.h, C.byref(ms)))
        return ms.value

    def download_hits(self, width, height, spp, want_tuv=True):
        shape = (height, width, spp)
        tri = np.empty(shape, np.uint32)
        t = np.empty(shape, np.float32) if want_tuv else None
        u = np.empty(shape, np.float32) if want_tuv else None
        v = np.empty(shape, np.float32) if want_tuv else None
        self._ck(self.lib.cuda_trace_download_hits(self.h, _p(tri, _U32P), _p(t, _F32P), _p(u, _F32P), _p(v, _F32P)))
        return tri, t, u, v

    def mailbox_stats(self):
        """-> (tests asked for, tests answered from the mailbox) of the last intersect_rays(..., mailbox=True)"""
        a, b = C.c_uint64(0), C.c_uint64(0)
        self._ck(self.lib.cuda_trace_mailbox_stats(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def intersect_rays(self, origins, dirs, variant=VARIANT_MT, mailbox=False):
        variant = variant | (0x100 if mailbox else 0)
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        n = len(o)
        tri, t, u, v = (np.empty(n, np.uint32), np.empty(n, np.float32), np.empty(n, np.float32),
                        np.empty(n, np.float32))
        self._ck(self.lib.cuda_trace_intersect_rays(self.h, n, _p(o, _F32P), _p(d, _F32P), variant,
                                                    _p(tri, _U32P), _p(t, _F32P), _p(u, _F32P), _p(v, _F32P)))
        return tri, t, u, v

    def query_rays(self, origins, dirs, t_max=None, occlusion=False, variant=VARIANT_MT, stream=None):
        """cuda_trace_query_rays on torch CUDA tensors: origins / dirs float32 (n, 3) on the context's first device,
        t_max None (unbounded), a float, or a float32 (n,) tensor.  Enqueued on ``stream`` (default: torch's current
        stream) without waiting; the outputs are allocated on that stream.  -> (tri int32 with -1 on a miss, t, u, v)
        for the closest hit, or a bool (n,) tensor for ``occlusion``."""
        import torch
        dev = torch.device("cuda", self.devices[0])

        def check(x, name, shape):
            if not isinstance(x, torch.Tensor):
                raise TypeError("%s must be a torch tensor" % name)
            if x.device != dev:
                raise ValueError("%s must be on %s (got %s)" % (name, dev, x.device))
            if x.dtype != torch.float32:
                raise TypeError("%s must be float32 (got %s)" % (name, x.dtype))
            if tuple(x.shape) != shape:
                raise ValueError("%s must have shape %s (got %s)" % (name, shape, tuple(x.shape)))
            return x.contiguous()

        if not isinstance(origins, torch.Tensor) or origins.dim() != 2:
            raise ValueError("origins must be a (n, 3) tensor")
        n = origins.shape[0]
        if n >= 2 ** 32:
            raise ValueError("at most 2^32 - 1 rays per query")
        stream = torch.cuda.current_stream(dev) if stream is None else stream
        with torch.cuda.stream(stream):
            o = check(origins, "origins", (n, 3))
            d = check(dirs, "dirs", (n, 3))
            b = RayBatch()
            b.n, b.variant = n, int(variant)
            b.kind = QUERY_OCCLUSION if occlusion else QUERY_CLOSEST
            b.origins, b.dirs = o.data_ptr(), d.data_ptr()
            tm = None
            if isinstance(t_max, torch.Tensor):
                tm = check(t_max, "t_max", (n,))
                b.t_max, b.t_max_all = tm.data_ptr(), float("inf")
            else:
                b.t_max, b.t_max_all = None, float("inf") if t_max is None else float(t_max)
            if occlusion:
                occ = torch.empty(n, dtype=torch.bool, device=dev)  # written as 0 / 1 bytes
                b.occluded = occ.data_ptr()
                out = occ
            else:
                tri = torch.empty(n, dtype=torch.int32, device=dev)
                t, u, v = (torch.empty(n, dtype=torch.float32, device=dev) for _ in range(3))
                b.tri_idx, b.t, b.u, b.v = tri.data_ptr(), t.data_ptr(), u.data_ptr(), v.data_ptr()
                out = (tri, t, u, v)
            # torch's default stream is the legacy NULL stream, which the C call would read as "the context's
            # stream": name it as cudaStreamLegacy (0x1) instead
            self._ck(self.lib.cuda_trace_query_rays(self.h, C.byref(b), C.c_void_p(stream.cuda_stream or 1)))
        return out

    def intersect_rays_brute_force(self, origins, dirs):
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        n = len(o)
        tri, t, u, v = (np.empty(n, np.uint32), np.empty(n, np.float32), np.empty(n, np.float32),
                        np.empty(n, np.float32))
        self._ck(self.lib.cuda_trace_intersect_rays_brute_force(self.h, n, _p(o, _F32P), _p(d, _F32P), _p(tri, _U32P),
                                                                _p(t, _F32P), _p(u, _F32P), _p(v, _F32P)))
        return tri, t, u, v

    def last_call_timing(self):
        """ms since the entry of the last trace_tiles call: submitted, traced, copied, returned, prepared,
        launching, launched."""
        ms = (C.c_double * 7)()
        self._ck(self.lib.cuda_trace_last_call_timing(self.h, ms))
        return [float(x) for x in ms]

    def strip_cycles(self):
        """SM cycles per strip of the last frame (this shard's order); empty when cost recording was off."""
        n = C.c_uint64(0)
        self._ck(self.lib.cuda_trace_download_strip_cycles(self.h, None, 0, C.byref(n)))
        out = np.zeros(n.value, np.uint32)
        if n.value:
            self._ck(self.lib.cuda_trace_download_strip_cycles(self.h, _p(out, _U32P), n.value, C.byref(n)))
        return out

    def ray_march(self, origins, dirs):
        o = np.ascontiguousarray(origins, np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, np.float32).reshape(-1, 3)
        n = len(o)
        hit, t = np.empty(n, np.uint32), np.empty(n, np.float32)
        self._ck(self.lib.cuda_trace_ray_march(self.h, n, _p(o, _F32P), _p(d, _F32P), _p(hit, _U32P), _p(t, _F32P)))
        return hit, t

    def sample_table(self, spp):
        xy = np.zeros((spp, 2), np.float32)
        self._ck(self.lib.cuda_trace_sample_table(self.h, spp, _p(xy, _F32P)))
        return xy

    # -- QMC sample tables (the reference's sampling module)
    QMC_KINDS = {"halton": 0, "hammersley": 1, "halton_zaremba": 2, "hammersley_zaremba": 3, "base2": 4, "sobol": 5,
                 "larcher_pillichshammer": 6}
    QMC_SCRAMBLES = {"none": 0, "braaten_weller": 1, "faure": 2, "reverse": 3, "custom": 4}

    def qmc_sequence(self, kind, n_begin, count, dim_begin=0, dim_count=1, num_smp=1, bits=0, scramble="none",
                     perm=None, perm_primes=0):
        """-> float64 [count, dim_count].  scramble "braaten_weller" loads assets/sampling/braaten_weller_16.u32
        unless ``perm`` is given; "custom" needs ``perm`` (tables of the first ``perm_primes`` primes back to back)."""
        k, s = self.QMC_KINDS[kind], self.QMC_SCRAMBLES[scramble]
        if s == 1 and perm is None:
            path = os.path.join(os.path.dirname(PKG), "assets", "sampling", "braaten_weller_16.u32")
            perm, perm_primes = np.fromfile(path, np.uint32), 16
        if perm is not None:
            perm = np.ascontiguousarray(perm, np.uint32)
        out = np.zeros((count, dim_count), np.float64)
        self._ck(self.lib.cuda_trace_qmc_sequence(self.h, k, s, _p(perm, _U32P), perm_primes, n_begin, count, dim_begin,
                                                  dim_count, num_smp, bits, out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def qmc_cranley_patterson(self, x, e):
        x = np.ascontiguousarray(x, np.float64)
        out = np.zeros_like(x)
        self._ck(self.lib.cuda_trace_qmc_cranley_patterson(self.h, x.ctypes.data_as(C.POINTER(C.c_double)), float(e),
                                                           x.size, out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def set_counting(self, enable):
        self._ck(self.lib.cuda_trace_set_counting(self.h, int(enable)))

    def get_counters(self):
        c = CountersC()
        self._ck(self.lib.cuda_trace_get_counters(self.h, C.byref(c)))
        return dict(rays=int(c.rays), cells=int(c.cells), tri_tests=int(c.tri_tests), hits=int(c.hits))

    def flush_l2(self):
        """Measurement helper (libcuda_trace_measure.so, not the product library): evict L2 on this context's devices."""
        self.sync()
        for dev in self.devices:
            flush_l2(dev)

    def kernel_launches(self):
        return int(self.lib.cuda_trace_kernel_launches(self.h))

    def set_shard(self, rank, world):
        self._ck(self.lib.cuda_trace_set_shard(self.h, rank, world))

    def set_shard_signals(self, enable):
        self._ck(self.lib.cuda_trace_set_shard_signals(self.h, int(enable)))

    def prepare_framebuffer(self, width, height):
        self._ck(self.lib.cuda_trace_prepare_framebuffer(self.h, width, height))

    def export_framebuffer(self):
        buf = C.create_string_buffer(64)
        self._ck(self.lib.cuda_trace_export_framebuffer(self.h, buf))
        return buf.raw

    def import_framebuffer(self, handle, width, height):
        buf = C.create_string_buffer(bytes(handle), 64)
        self._ck(self.lib.cuda_trace_import_framebuffer(self.h, buf, width, height))

    def framebuffer_device_ptr(self):
        return self.lib.cuda_trace_framebuffer_device_ptr(self.h)

    def stream(self):
        return self.lib.cuda_trace_stream(self.h)
