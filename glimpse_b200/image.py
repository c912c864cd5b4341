"""Frame holders: ``Image`` (photograph + per-frame Camera) and ``Raster`` (DEM / viewshed grid, or an
orthoimage with a datetime that an ``Observer`` tracks through like an ``Image``).

Mirrors the parts of reference ``image.py:86-119,137-214,279-299`` and ``raster.py:30-421,891-1027``
that the Tracker touches.  File decoding is host I/O and out of scope; in-memory arrays are the
norm (``img.array = ndarray``), with an OpenCV read as a convenience when a path exists.
"""
from __future__ import annotations

import datetime as _dt
import os
from typing import Iterable, Optional, Union

import numpy as np

from . import _lib
from .camera import Camera


def decode_jpeg(data: bytes, gray: bool = None):
    """JPEG bytes -> uint8 tensor on the current device, (rows, columns, 3) RGB or (rows, columns) luma (``gray``; default: as the
    stream is encoded), decoded by nvJPEG through ``gb_decode_jpeg``."""
    import ctypes as C

    torch = _lib.require_cuda()
    lib = _lib.load()
    w, h, c = C.c_int32(), C.c_int32(), C.c_int32()
    _lib.check(lib.gb_jpeg_info(data, len(data), C.byref(w), C.byref(h), C.byref(c)))
    bands = 1 if (gray or (gray is None and c.value == 1)) else 3
    dev = torch.device("cuda", torch.cuda.current_device())
    out = torch.empty((h.value, w.value, bands) if bands == 3 else (h.value, w.value), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    _lib.check(lib.gb_decode_jpeg(data, len(data), w.value, h.value, bands, out.data_ptr(), stream.cuda_stream))
    stream.synchronize()  # (the bytes object must outlive the decode)
    return out


class Image:
    """Photograph taken by a :class:`Camera` at a known time (reference ``image.py:17-119``)."""

    def __init__(self, path, cam: Union[dict, Camera] = None, datetime: _dt.datetime = None, exif=None) -> None:
        self.path = str(path)
        if isinstance(cam, dict):
            cam = Camera(**cam)
        if cam is None:
            raise ValueError("Image needs a Camera (EXIF parsing is out of scope)")
        if datetime is None:
            raise ValueError("Image needs a datetime (EXIF parsing is out of scope)")
        self.cam = cam
        self.datetime = datetime
        self.exif = exif
        self.array: Optional[np.ndarray] = None
        self.device_array = None  # the frame in device memory (read_device)

    @property
    def size(self) -> np.ndarray:
        return self.cam.imgsz

    def read(self, box: Iterable[int] = None, cache: bool = True) -> np.ndarray:
        """Pixel array, optionally cropped to (left, top, right, bottom) (reference image.py:137-214)."""
        array = self.array
        if array is None:
            if not os.path.exists(self.path):
                raise FileNotFoundError(f"{self.path}: set Image.array or give a readable path")
            import cv2

            array = cv2.imread(self.path, cv2.IMREAD_UNCHANGED)
            if array is None:
                raise IOError(f"Could not decode {self.path}")
            if array.ndim == 3:
                array = array[:, :, ::-1]
            w, h = (int(v) for v in self.cam.imgsz)
            if (array.shape[1], array.shape[0]) != (w, h):
                array = cv2.resize(array, (w, h), interpolation=cv2.INTER_AREA)
            array = np.ascontiguousarray(array)
            if cache:
                self.array = array
        if box is not None:
            array = array[box[1]:box[3], box[0]:box[2]]
        return array

    def read_device(self, cache: bool = True):
        """The image as a uint8 tensor in device memory, decoded there from its JPEG file by nvJPEG (``gb_decode_jpeg``; the
        reference decodes on the host through GDAL, image.py:137-214): (rows, columns, 3) RGB or (rows, columns) for a grey file.
        With ``cache`` it is kept in ``device_array`` and a Tracker reads the frame from there instead of uploading ``array``.
        Decoders differ in the last grey levels (IDCT, chroma upsampling): use ``read`` / ``array`` where the exact pixels of one
        decoder matter.  The file must have the camera's image size (no resampling on the way)."""
        held = getattr(self, "device_array", None)
        if held is not None:
            return held
        with open(self.path, "rb") as f:
            data = f.read()
        tensor = decode_jpeg(data)
        w, h = (int(v) for v in self.cam.imgsz)
        if (tensor.shape[1], tensor.shape[0]) != (w, h):
            raise NotImplementedError(f"{self.path}: {tensor.shape[1]} x {tensor.shape[0]} pixels, the camera has {w} x {h} "
                                      "(resampling while decoding is not implemented: use read())")
        if cache:
            self.device_array = tensor
        return tensor

    def project(self, cam: Camera, method: str = "linear") -> np.ndarray:
        """Project the image into another camera at the same position (reference image.py:301-361): (cam.imgsz[1],
        cam.imgsz[0], bands) of the image's pixel type, NaN (0 in an integer image) where the target sees nothing of the
        source.  One thread per target pixel on the device (``gb_project_image``)."""
        import ctypes as C

        from .camera import lower_camera
        from .session import device_frame

        if method not in ("linear", "nearest"):
            raise ValueError(f"Method '{method}' is not defined")
        if not all(np.asarray(cam.xyz) == np.asarray(self.cam.xyz)):
            raise ValueError("Source and target cameras have different positions ('xyz')")
        torch = _lib.require_cuda()
        lib = _lib.load()
        array = self.read()
        frame = device_frame(array)  # uint8 / uint16 / float32 / float64 as they are, other types as NumPy promotes them
        dev = torch.device("cuda", torch.cuda.current_device())
        pixels = torch.from_numpy(frame.reshape(-1).view(np.uint8)).to(dev)  # (bytes: the frame keeps its own pixel type)
        src = _lib.gb_image()
        src.pixels = pixels.data_ptr()
        src.width, src.height, src.pitch = frame.shape[1], frame.shape[0], frame.strides[0]
        src.nchan = 1 if frame.ndim == 2 else frame.shape[2]
        src.dtype = _lib.GB_PIX[frame.dtype.name]
        src.cam = lower_camera(self.cam)
        dst = lower_camera(cam)
        w, h = (int(v) for v in cam.imgsz)
        out = torch.empty(h * w * src.nchan * frame.dtype.itemsize, dtype=torch.uint8, device=dev)
        _lib.check(lib.gb_project_image(C.byref(src), C.byref(dst), 1 if method == "linear" else 0, out.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream))
        result = out.cpu().numpy().view(frame.dtype).reshape(h, w, src.nchan)
        if result.dtype != array.dtype:  # a type the device holds promoted: back to the image's own, as the reference assigns it
            with np.errstate(invalid="ignore"):
                result = result.astype(array.dtype)
        return result

    def xyz_to_uv(self, xyz, **kwargs):
        return self.cam.xyz_to_uv(xyz, **kwargs)

    def uv_to_xyz(self, uv, directions: bool = False, **kwargs):
        return self.cam.uv_to_xyz(uv, directions=directions, **kwargs)

    def inbounds(self, uv):
        return self.cam.inframe(uv)


class Raster:
    """Regular grid of values (reference ``raster.py:523-560``): DEM, DEM uncertainty, viewshed — or, with a
    ``datetime``, one frame of an Observer made of orthoimages (the reference Tracker only needs ``xyz_to_uv``,
    ``inbounds``, ``size`` and ``read`` of a frame: tracker.py:580-607, observer.py:115-130).

    ``x`` / ``y`` are the outer limits (left, right) / (top, bottom) or cell-centre vectors, exactly
    as the reference accepts them; a scalar ``array`` is the constant surface the motion models build
    from numbers (reference ``track/motion.py:136-141``).
    """

    def __init__(self, array, x=None, y=None, datetime: _dt.datetime = None) -> None:
        # values keep their type (an orthoimage is tracked in the type it has, like Image.array); surfaces are lowered as float64
        self.array = np.atleast_2d(np.asarray(array)) if np.ndim(array) else np.asarray(array, dtype=float)
        self.datetime = datetime
        shape = self.array.shape[0:2] if self.array.ndim >= 2 else (1, 1)
        self.xlim = self._limits(x, shape[1])
        self.ylim = self._limits(y, shape[0])
        # identity used to share one device surface between equal constant rasters
        # (a string: its hash is computed once, and a thousand models each wrap the same number into a raster of their own)
        self._const_key = ("const|%r|%r|%r" % (float(self.array.flat[0]), tuple(self.xlim.tolist()), tuple(self.ylim.tolist()))
                           if self.constant else None)

    @staticmethod
    def _limits(value, n) -> np.ndarray:
        if value is None:
            return np.array((0.0, float(n)))
        value = np.atleast_1d(np.asarray(value, dtype=float))
        if value.size > 2:  # cell centres
            d = value[1] - value[0]
            return np.array((value[0] - d / 2, value[-1] + d / 2))
        return value.astype(float)

    @property
    def size(self) -> np.ndarray:
        if self.array.ndim < 2:
            return np.array((1, 1))
        return np.array(self.array.shape[0:2][::-1])

    @property
    def d(self) -> np.ndarray:
        """Signed cell size (dx, dy) (reference raster.py:119-122)."""
        return np.hstack((np.diff(self.xlim), np.diff(self.ylim))) / self.size

    def xyz_to_uv(self, xyz) -> np.ndarray:
        """World -> image coordinates of the grid; z is optional and unused (reference raster.py:423-445)."""
        xyz = np.asarray(xyz)
        return (xyz[:, 0:2] - (self.xlim[0], self.ylim[0])) / self.d

    def uv_to_xyz(self, uv) -> np.ndarray:
        """Image -> world coordinates, z = NaN (reference raster.py:447-459)."""
        uv = np.asarray(uv)
        xy = uv * self.d + (self.xlim[0], self.ylim[0])
        return np.column_stack((xy, np.full((xy.shape[0], 1), np.nan)))

    def inbounds(self, uv) -> np.ndarray:
        """Whether image coordinates are in or on the bounds (reference raster.py:339-341)."""
        uv = np.asarray(uv)
        return np.all((uv >= 0) & (uv <= self.size), axis=1)

    def read(self, box: Iterable[int] = None, cache: bool = True) -> np.ndarray:
        """Values, optionally cropped to (left, top, right, bottom) (reference raster.py:763-836; in-memory arrays only)."""
        if box is None:
            return self.array
        box = np.asarray(box).reshape(-1, 2)
        if not np.issubdtype(box.dtype, np.integer):
            raise ValueError("Box must be integers")
        if not np.all(self.inbounds(box)):
            raise ValueError("Box is out of bounds")
        return self.array[box[0, 1]:box[1, 1], box[0, 0]:box[1, 0]]

    @property
    def x(self) -> np.ndarray:
        """Cell-centre x coordinates in array order (reference raster.py:139-156)."""
        return self._centres(self.xlim, self.size[0])

    @property
    def y(self) -> np.ndarray:
        """Cell-centre y coordinates in array order (reference raster.py:161-174)."""
        return self._centres(self.ylim, self.size[1])

    @staticmethod
    def _centres(lim, n) -> np.ndarray:
        half = abs((lim[1] - lim[0]) / n) / 2
        value = np.linspace(start=min(lim) + half, stop=max(lim) - half, num=int(n))
        return value[::-1] if lim[1] < lim[0] else value

    def viewshed(self, origin, correction=False) -> np.ndarray:
        """Boolean array of the cells visible from ``origin`` (x, y, z) (reference raster.py:1293-1389): rings of cells by
        rounded distance, swept outwards on the device against the previous ring's interpolated horizon (``gb_viewshed``).
        ``correction``: arguments of ``helpers.elevation_corrections`` (``radius``, ``refraction``), ``True`` for its
        defaults, or ``False`` / ``None``."""
        import ctypes as C
        import warnings

        d = np.abs(self.d)
        if not all(d[0] == d):
            warnings.warn("DEM cells not square " + str(tuple(d)) + " - may lead to unexpected results")
        origin = np.asarray(origin, dtype=float)
        if not (min(self.xlim) <= origin[0] <= max(self.xlim) and min(self.ylim) <= origin[1] <= max(self.ylim)):
            warnings.warn("Origin not in DEM - may lead to unexpected results")
        if correction is True:
            correction = {}
        corr = None
        if isinstance(correction, dict):
            corr = (C.c_double * 2)(float(correction.get("radius", 6.3781e6)), float(correction.get("refraction", 0.13)))
        torch = _lib.require_cuda()
        lib = _lib.load()
        dev = torch.device("cuda", torch.cuda.current_device())
        z = np.ascontiguousarray(self.array, dtype=float)
        ny, nx = z.shape
        x, y = self.x, self.y
        # rings between the nearest and the farthest cell: from the bounding box of the cell centres
        near = np.hypot(np.clip(origin[0], x.min(), x.max()) - origin[0], np.clip(origin[1], y.min(), y.max()) - origin[1])
        far = max(np.hypot(cx - origin[0], cy - origin[1]) for cx in (x.min(), x.max()) for cy in (y.min(), y.max()))
        max_rings = int(far / d[0]) - int(near / d[0]) + 4
        nbytes = int(lib.gb_viewshed_work_bytes(nx, ny, max_rings))
        work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        z_d, x_d, y_d = (torch.from_numpy(np.array(v, dtype=float, order="C", copy=True)).to(dev) for v in (z, x, y))
        out = torch.empty(ny * nx, dtype=torch.uint8, device=dev)
        _lib.check(lib.gb_viewshed(z_d.data_ptr(), nx, ny, x_d.data_ptr(), y_d.data_ptr(), float(d[0]), (C.c_double * 3)(*origin[:3]),
                                   corr, max_rings, work.data_ptr(), nbytes, out.data_ptr(), torch.cuda.current_stream().cuda_stream))
        status = int(work[:4].cpu().numpy().view(np.int32)[0])  # (synchronises)
        if status != 0:
            raise RuntimeError(f"viewshed: device status {status}")
        return out.cpu().numpy().reshape(ny, nx).astype(bool)

    def lower_grid_camera(self) -> "_lib.gb_camera":
        """The frame's world -> image map as an affine ``gb_camera`` (``affine = 1``: origin in ``xyz``, cell size in ``f``)."""
        out = _lib.gb_camera()
        d = self.d
        out.affine = 1
        out.xyz[:] = [float(self.xlim[0]), float(self.ylim[0]), 0.0]
        out.f[:] = [float(d[0]), float(d[1])]
        out.imgsz[:] = [int(v) for v in self.size]
        return out

    @property
    def constant(self) -> bool:
        return self.array.ndim < 2 or self.array.size == 1

    def lower_host(self) -> "tuple[_lib.gb_surface, object]":
        """-> (``gb_surface`` without its device pointer, the (nx, ny) array of cell values on increasing centres or None)."""
        s = _lib.gb_surface()
        s.xmin, s.xmax = float(min(self.xlim)), float(max(self.xlim))
        s.ymin, s.ymax = float(min(self.ylim)), float(max(self.ylim))
        if self.constant:
            s.z = None
            s.value = float(self.array.flat[0])
            return s, None
        ny, nx = self.array.shape
        dx = (self.xlim[1] - self.xlim[0]) / nx
        dy = (self.ylim[1] - self.ylim[0]) / ny
        z = self.array.T.astype(float, copy=False)  # (nx, ny)
        if dx < 0:
            z = z[::-1, :]
        if dy < 0:
            z = z[:, ::-1]
        if nx < 2 or ny < 2:
            raise NotImplementedError("1-D rasters are not supported on device")
        s.nx, s.ny = nx, ny
        s.dx, s.dy = abs(dx), abs(dy)
        s.x0, s.y0 = s.xmin + s.dx / 2, s.ymin + s.dy / 2
        s.value = 0.0
        return s, np.ascontiguousarray(z)

    def lower(self, torch, device) -> "tuple[_lib.gb_surface, object]":
        """-> (``gb_surface``, device tensor kept alive by the caller)."""
        s, z = self.lower_host()
        if z is None:
            return s, None
        tensor = torch.as_tensor(z).to(device)
        s.z = tensor.data_ptr()
        return s, tensor
