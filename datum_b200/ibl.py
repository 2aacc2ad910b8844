"""Python host side of the IBL bake: the reference's tools/ibl.h surface over the C ABI.

Function names, argument order and buffer conventions follow the reference
(paths relative to /root/reference):

    image_buildmips_cube_ibl(width, height, levels, bits)         tools/ibl.h:9
    image_pack_cube_ibl(image, width, height, levels, bits)       tools/ibl.h:11
    image_pack_envbrdf(width, height, bits)                       tools/ibl.h:13
    image_pack_watercolor(deep, shallow, depthscale, ...)         tools/ibl.h:15

`bits` is a caller-allocated uint32 buffer of image_datasize(width, height, 6,
levels) bytes (tools/assetbuilder.cpp:439, 484), level 0 pre-filled where the
reference expects it, written in place.  numpy arrays and (pinned) CPU torch
tensors are accepted.  All arithmetic happens in libdatum_ibl_cuda.
"""

import atexit
import ctypes
import sys
import weakref

import numpy as np

from . import _lib

FORMAT_RGBE = 0
FORMAT_F32 = 1
FORMAT_F16 = 2

# bytes per texel of each format
TEXEL_BYTES = {FORMAT_RGBE: 4, FORMAT_F32: 16, FORMAT_F16: 8}

# element dtype of the float chain formats (4 channels per texel)
_FLOAT_DTYPES = {FORMAT_F32: np.float32, FORMAT_F16: np.float16}


class IblError(RuntimeError):
    """Raised for every non-zero status of the C ABI (the reference functions are void)."""


def image_maxlevels(width, height):
    """tools/assetpacker.cpp:472-484"""
    levels = 1
    for i in range(16):
        if (width >> i) == 1 or (height >> i) == 1:
            break
        levels += 1
    return levels


def image_datasize(width, height, layers, levels):
    """tools/assetpacker.cpp:488-497 (bytes)"""
    return sum((width >> i) * (height >> i) * layers * 4 for i in range(levels))


def level_offsets(width, height, levels, layers=6):
    """Word offset of every level inside a chain payload, plus the total (levels + 1 entries)."""
    offsets = [0]
    for i in range(levels):
        offsets.append(offsets[-1] + (width >> i) * (height >> i) * layers)
    return offsets


def float_chain_texels(width, height, levels):
    """Texels of a float chain: the same levels as image_datasize, 4 channels each."""
    return sum((width >> i) * (height >> i) * 6 for i in range(levels))


def _texel_bytes(fmt):
    if fmt not in TEXEL_BYTES:
        raise ValueError("unknown texel format %r" % (fmt,))
    return TEXEL_BYTES[fmt]


def _float_dtype(fmt):
    if fmt not in _FLOAT_DTYPES:
        raise ValueError("unknown float chain format %r (FORMAT_F32 or FORMAT_F16)" % (fmt,))
    return np.dtype(_FLOAT_DTYPES[fmt])


def _check_dtype(buf, dtype, what):
    """A numpy array or a torch tensor of exactly `dtype` (numpy dtype)."""
    got = buf.dtype if isinstance(buf, np.ndarray) else getattr(buf, "dtype", None)
    if isinstance(buf, np.ndarray):
        ok = got == dtype
    else:
        import torch
        ok = got == {np.dtype(np.float32): torch.float32, np.dtype(np.float16): torch.float16}[dtype]
    if not ok:
        raise ValueError("%s must hold %s texels, not %s" % (what, dtype.name, got))


def _float_chain_pointers(fmt, width, height, levels, chains):
    """ctypes array of the host chains of a float batch, every one checked for dtype and size."""
    dtype = _float_dtype(fmt)
    need = float_chain_texels(width, height, levels) * _texel_bytes(fmt)
    pointers = (ctypes.c_void_p * max(len(chains), 1))()
    for i, chain in enumerate(chains):
        what = "chains[%d]" % i
        if hasattr(chain, "is_cuda") and chain.is_cuda:
            raise ValueError("%s must be a host buffer" % what)
        _check_dtype(chain, dtype, what)
        pointers[i] = _host_pointer(chain, need, what)
    return pointers


def _host_pointer(buf, min_bytes, what):
    """Address of a writable, contiguous host buffer (numpy array or CPU torch tensor)."""
    if isinstance(buf, np.ndarray):
        if not buf.flags["C_CONTIGUOUS"]:
            raise ValueError("%s must be C-contiguous" % what)
        if buf.nbytes < min_bytes:
            raise ValueError("%s holds %d bytes, %d needed" % (what, buf.nbytes, min_bytes))
        return buf.ctypes.data
    if hasattr(buf, "data_ptr"):  # torch tensor
        if buf.is_cuda:
            raise ValueError("%s must be a host buffer" % what)
        if not buf.is_contiguous():
            raise ValueError("%s must be contiguous" % what)
        if buf.numel() * buf.element_size() < min_bytes:
            raise ValueError("%s holds %d bytes, %d needed" % (what, buf.numel() * buf.element_size(), min_bytes))
        return buf.data_ptr()
    raise TypeError("%s must be a numpy array or a torch tensor" % what)


def _float_host_buffer(fmt, buf, texels, what):
    """Address of a host buffer of `texels` texels of float format `fmt`, checked for dtype and size."""
    if hasattr(buf, "is_cuda") and buf.is_cuda:
        raise ValueError("%s must be a host buffer" % what)
    _check_dtype(buf, _float_dtype(fmt), what)
    return _host_pointer(buf, texels * _texel_bytes(fmt), what)


def _equirect_image(image):
    image = np.ascontiguousarray(image, dtype=np.float32)
    if image.ndim != 3 or image.shape[2] != 4:
        raise ValueError("image must be (H, W, 4) float32")
    return image


def _face_images(faces):
    faces = np.ascontiguousarray(faces, dtype=np.uint32)
    if faces.ndim != 3 or faces.shape[0] != 6:
        raise ValueError("faces must be (6, H, W) uint32")
    return faces


def _device_pointer(t, min_bytes, what, device):
    if t is None:
        return None
    if not (hasattr(t, "is_cuda") and t.is_cuda):
        raise ValueError("%s must be a CUDA tensor" % what)
    if t.device.index != device:
        raise ValueError("%s lives on cuda:%s, the context is bound to cuda:%d" % (what, t.device.index, device))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % what)
    if t.numel() * t.element_size() < min_bytes:
        raise ValueError("%s holds %d bytes, %d needed" % (what, t.numel() * t.element_size(), min_bytes))
    return t.data_ptr()


class IblContext:
    """One bake context bound to one CUDA device (wraps datum_ibl_ctx)."""

    def __init__(self, device=0):
        self._lib = _lib.load()
        handle = ctypes.c_void_p()
        if self._lib.datum_ibl_create(int(device), ctypes.byref(handle)):
            raise IblError(self._error())
        self._handle = handle
        self.device = int(device)
        self._torch_stream = None
        _live.add(self)

    # ---- plumbing ----

    def _error(self):
        return self._lib.datum_ibl_last_error().decode("utf-8", "replace")

    def _check(self, status):
        if status:
            raise IblError(self._error())

    def close(self):
        if getattr(self, "_handle", None):
            self._lib.datum_ibl_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            if not sys.is_finalizing():
                self.close()
        except Exception:
            pass

    def __hash__(self):
        return id(self)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def stream_pointer(self):
        return self._lib.datum_ibl_stream(self._handle)

    def torch_stream(self):
        """The context's CUDA stream as a torch stream: torch work issued under
        `with torch.cuda.stream(ctx.torch_stream())` is ordered with the kernels."""
        if self._torch_stream is None:
            import torch
            self._torch_stream = torch.cuda.ExternalStream(self.stream_pointer, device=torch.device("cuda", self.device))
        return self._torch_stream

    def synchronize(self):
        self._check(self._lib.datum_ibl_synchronize(self._handle))

    def _after_torch(self):
        """The context's stream is its own (non-blocking) stream: before a *_device entry point reads or
        writes caller tensors, make it wait for whatever torch has queued on its CURRENT stream (the
        producers of those tensors: a torch.zeros, a copy_, ...).  Free when the caller already works
        under `with torch.cuda.stream(ctx.torch_stream())`."""
        import torch
        current = torch.cuda.current_stream(self.device)
        if current.cuda_stream != self.stream_pointer:
            self.torch_stream().wait_event(current.record_event())

    @property
    def launch_count(self):
        return int(self._lib.datum_ibl_launch_count(self._handle))

    def set_prefilter_variant(self, variant):
        self._check(self._lib.datum_ibl_set_prefilter_variant(self._handle, int(variant)))

    def set_tuning(self, key, value):
        """Development knobs of datum_ibl_set_tuning (A/B timing)."""
        self._check(self._lib.datum_ibl_set_tuning(self._handle, key.encode(), int(value)))

    def last_prefilter_ms(self):
        ms = ctypes.c_float()
        self._check(self._lib.datum_ibl_last_prefilter_ms(self._handle, ctypes.byref(ms)))
        return float(ms.value)

    def dominant_kernel_stats(self, reset=True):
        """(launches, mean ms, texel-samples per launch) of the level-1 prefilter launches since the last reset."""
        n, ms, ts = ctypes.c_int(), ctypes.c_double(), ctypes.c_double()
        self._check(self._lib.datum_ibl_dominant_kernel_stats(self._handle, 1 if reset else 0, ctypes.byref(n), ctypes.byref(ms), ctypes.byref(ts)))
        return int(n.value), float(ms.value), float(ts.value)

    def measure_fp32_peak(self):
        """FP32 FMA throughput of the device in TFLOP/s (register-resident FFMA chains)."""
        tflops = ctypes.c_double()
        self._check(self._lib.datum_ibl_measure_fp32_peak(self._handle, ctypes.byref(tflops)))
        return float(tflops.value)

    def measure_fp32x2_peak(self):
        """Same, issued as packed fma.rn.f32x2 (FFMA2)."""
        tflops = ctypes.c_double()
        self._check(self._lib.datum_ibl_measure_fp32x2_peak(self._handle, ctypes.byref(tflops)))
        return float(tflops.value)

    # ---- prefilter chain: tools/ibl.cpp:242-279 ----

    def image_buildmips_cube_ibl(self, width, height, levels, bits, samples=1024):
        """Host payload, level 0 pre-filled, levels >= 1 written in place (tools/ibl.h:9)."""
        ptr = _host_pointer(bits, image_datasize(width, height, 6, levels), "bits")
        self._check(self._lib.datum_ibl_buildmips_cube_ibl(self._handle, width, height, levels, samples, ptr))

    def bake_probes(self, width, height, levels, payloads, samples=1024, sh9=False):
        """A batch of independent bakes (datum_ibl_bake_probes): every payload is a host array used
        like the `bits` of image_buildmips_cube_ibl; uploads, kernels and downloads of consecutive
        probes overlap (fully when the payloads are pinned).  With sh9=True returns the SH9
        projection of every level 0 as a (count, 9, 3) float32 array."""
        count = len(payloads)
        need = image_datasize(width, height, 6, levels)
        pointers = (ctypes.c_void_p * max(count, 1))()
        for i, payload in enumerate(payloads):
            pointers[i] = _host_pointer(payload, need, "payloads[%d]" % i)
        sh = np.zeros((count, 9, 3), np.float32) if sh9 else None
        self._check(self._lib.datum_ibl_bake_probes(self._handle, count, width, height, levels, samples, pointers, sh.ctypes.data if sh9 and count else None))
        return sh

    def buildmips_cube_ibl_device(self, width, height, levels, d_bits, samples=1024, d_f32=None):
        """Same chain on a device-resident payload (int32/uint32 CUDA tensor); asynchronous on the
        context's stream, ordered BEHIND the work torch has queued on its current stream; results are
        ready after ctx.synchronize() (or for torch work issued under ctx.torch_stream()).
        d_f32: optional float32 CUDA tensor receiving the pre-quantisation rgb of levels >= 1."""
        total = image_datasize(width, height, 6, levels)
        level0 = width * height * 6 * 4
        bits_ptr = _device_pointer(d_bits, total, "d_bits", self.device)
        f32_ptr = _device_pointer(d_f32, (total - level0) * 3, "d_f32", self.device)
        self._after_torch()
        self._check(self._lib.datum_ibl_buildmips_cube_ibl_device(self._handle, width, height, levels, samples, bits_ptr, f32_ptr))

    def prefilter_level_device(self, d_src, ws, hs, level, levels, samples, row_begin, row_end, d_dst_words=None, d_dst_f32=None):
        """One level, rows [row_begin,row_end) of the 6*(hs/2) destination rows; asynchronous."""
        out_texels = 6 * (ws >> 1) * (hs >> 1)
        src_ptr = _device_pointer(d_src, 6 * ws * hs * 4, "d_src", self.device)
        words_ptr = _device_pointer(d_dst_words, out_texels * 4, "d_dst_words", self.device)
        f32_ptr = _device_pointer(d_dst_f32, out_texels * 12, "d_dst_f32", self.device)
        self._after_torch()
        self._check(self._lib.datum_ibl_prefilter_level_device(self._handle, src_ptr, ws, hs, level, levels, samples, row_begin, row_end, words_ptr, f32_ptr))

    # ---- float chains (RGBA32F / RGBA16F): the same chain without rgbe re-quantisation ----

    def buildmips_cube_float(self, fmt, width, height, levels, chain, samples=1024):
        """Host float chain (numpy array or CPU torch tensor: float32 for FORMAT_F32, float16 for
        FORMAT_F16, 4 channels per texel, the levels of image_datasize), level 0 pre-filled, levels >= 1
        written in place.  Synchronous."""
        if not (hasattr(chain, "is_cuda") and chain.is_cuda):
            _check_dtype(chain, _float_dtype(fmt), "chain")
        ptr = _host_pointer(chain, float_chain_texels(width, height, levels) * _texel_bytes(fmt), "chain")
        self._check(self._lib.datum_ibl_buildmips_cube_float(self._handle, fmt, width, height, levels, samples, ptr))

    def bake_probes_float(self, fmt, width, height, levels, chains, samples=1024, sh9=False):
        """A batch of float chains (datum_ibl_bake_probes_float): every chain is a host array of the format's
        dtype used like the `chain` of buildmips_cube_float, and ends with the same bytes; small probes share
        launches, and uploads, kernels and downloads of consecutive probes overlap (fully when the chains are
        pinned).  With sh9=True returns the SH9 projection of every level 0 as a (count, 9, 3) float32 array."""
        count = len(chains)
        pointers = _float_chain_pointers(fmt, width, height, levels, chains)
        sh = np.zeros((count, 9, 3), np.float32) if sh9 else None
        self._check(self._lib.datum_ibl_bake_probes_float(self._handle, fmt, count, width, height, levels, samples, pointers, sh.ctypes.data if sh9 and count else None))
        return sh

    def buildmips_cube_float_device(self, fmt, width, height, levels, d_chain, samples=1024, d_f32=None):
        """The same chain on a device-resident CUDA tensor of the format's dtype; asynchronous on the
        context's stream, ordered behind the work torch has queued on its current stream.  d_f32: optional
        float32 CUDA tensor receiving the fp32 rgb of levels >= 1 before rounding."""
        _check_dtype(d_chain, _float_dtype(fmt), "d_chain")
        texels = float_chain_texels(width, height, levels)
        chain_ptr = _device_pointer(d_chain, texels * _texel_bytes(fmt), "d_chain", self.device)
        if d_f32 is not None:
            _check_dtype(d_f32, np.dtype(np.float32), "d_f32")
        f32_ptr = _device_pointer(d_f32, (texels - 6 * width * height) * 12, "d_f32", self.device)
        self._after_torch()
        self._check(self._lib.datum_ibl_buildmips_cube_float_device(self._handle, fmt, width, height, levels, samples, chain_ptr, f32_ptr))

    def prefilter_level_float_device(self, fmt, d_src, ws, hs, level, levels, samples, row_begin, row_end, d_dst, d_dst_f32=None):
        """One level of a float chain, rows [row_begin,row_end) of the 6*(hs/2) destination rows; CUDA
        tensors of the format's dtype; asynchronous."""
        dtype = _float_dtype(fmt)
        _check_dtype(d_src, dtype, "d_src")
        _check_dtype(d_dst, dtype, "d_dst")
        if d_dst_f32 is not None:
            _check_dtype(d_dst_f32, np.dtype(np.float32), "d_dst_f32")
        out_texels = 6 * (ws >> 1) * (hs >> 1)
        src_ptr = _device_pointer(d_src, 6 * ws * hs * _texel_bytes(fmt), "d_src", self.device)
        dst_ptr = _device_pointer(d_dst, out_texels * _texel_bytes(fmt), "d_dst", self.device)
        f32_ptr = _device_pointer(d_dst_f32, out_texels * 12, "d_dst_f32", self.device)
        self._after_torch()
        self._check(self._lib.datum_ibl_prefilter_level_float_device(self._handle, fmt, src_ptr, ws, hs, level, levels, samples, row_begin, row_end, dst_ptr, f32_ptr))

    # ---- SH9: data/project.comp:23-106 ----

    # ---- one probe shared by the GPUs of a node: peer-mapped payloads, NVLink stores from the kernel epilogue ----

    def peer_alloc(self, nbytes):
        """Zeroed device memory other processes of the node can map.  Returns (address, 64-byte IPC handle)."""
        ptr = ctypes.c_void_p()
        handle = ctypes.create_string_buffer(64)
        self._check(self._lib.datum_ibl_peer_alloc(self._handle, nbytes, ctypes.byref(ptr), handle))
        return int(ptr.value), bytes(handle.raw)

    def peer_free(self, address):
        self._check(self._lib.datum_ibl_peer_free(self._handle, ctypes.c_void_p(address)))

    def peer_open(self, handle):
        """Map a peer's allocation (its 64-byte IPC handle) into this process; returns the local address."""
        ptr = ctypes.c_void_p()
        buf = ctypes.create_string_buffer(bytes(handle), 64)
        self._check(self._lib.datum_ibl_peer_open(self._handle, buf, ctypes.byref(ptr)))
        return int(ptr.value)

    def peer_close(self, address):
        self._check(self._lib.datum_ibl_peer_close(self._handle, ctypes.c_void_p(address)))

    def prefilter_level_peers(self, src_address, ws, hs, level, levels, samples, row_begin, row_end, rank, world, dst_addresses, flag_addresses=None, epoch=0):
        """prefilter_level_device on raw device addresses for rank `rank` of `world` GPUs sharing the probe:
        dst_addresses[r] = START of the destination level in rank r's payload as mapped here; every word of the
        slab goes to all of them.  With flag_addresses (flag blocks by rank) and epoch > 0 the launch signals
        the peers when it is complete and the stream then waits for theirs."""
        dst = (ctypes.c_void_p * world)(*dst_addresses)
        flags = (ctypes.c_void_p * world)(*flag_addresses) if flag_addresses is not None else None
        self._check(self._lib.datum_ibl_prefilter_level_peers(self._handle, ctypes.c_void_p(src_address), ws, hs, level, levels, samples, row_begin, row_end, rank, world, dst, flags, epoch))

    def prefilter_level_float_peers(self, fmt, src_address, ws, hs, level, levels, samples, row_begin, row_end, rank, world, dst_addresses, flag_addresses=None, epoch=0):
        """prefilter_level_peers for a float chain of format `fmt` (FORMAT_F32 or FORMAT_F16): raw device addresses,
        aligned to the texel size; every texel of the slab goes to the destination level of each rank's chain."""
        dst = (ctypes.c_void_p * world)(*dst_addresses)
        flags = (ctypes.c_void_p * world)(*flag_addresses) if flag_addresses is not None else None
        self._check(self._lib.datum_ibl_prefilter_level_float_peers(self._handle, fmt, ctypes.c_void_p(src_address), ws, hs, level, levels, samples, row_begin, row_end, rank, world, dst, flags, epoch))

    def peer_barrier(self, rank, world, flag_addresses, epoch):
        """Barrier of the GPUs sharing a probe, on the context's stream (flag blocks by rank)."""
        flags = (ctypes.c_void_p * world)(*flag_addresses)
        self._check(self._lib.datum_ibl_peer_barrier(self._handle, rank, world, flags, epoch))

    def set_peer_timeout_ms(self, milliseconds):
        """How long synchronize() lets the stream wait for a peer's arrival before it gives up (default 60 s)."""
        self._check(self._lib.datum_ibl_set_peer_timeout_ms(self._handle, int(milliseconds)))

    def sh9_partial_device(self, d_level0, fmt, width, height, row_begin, row_end, d_partial):
        """28 partial sums (27 coefficients + weight) into a float64 CUDA tensor; asynchronous."""
        texel_bytes = TEXEL_BYTES.get(fmt, 16)   # an unknown format is rejected by the C ABI
        src_ptr = _device_pointer(d_level0, 6 * width * height * texel_bytes, "d_level0", self.device)
        out_ptr = _device_pointer(d_partial, 28 * 8, "d_partial", self.device)
        self._after_torch()
        self._check(self._lib.datum_ibl_sh9_partial_device(self._handle, src_ptr, fmt, width, height, row_begin, row_end, out_ptr))

    def sh9_partial_peers(self, d_level0, fmt, width, height, row_begin, row_end, rank, world, slot_addresses, flag_addresses=None, epoch=0):
        """sh9_partial_device whose 28 sums also go to row [rank] of every peer's (world x 28) float64 array
        (addresses by rank, peer_alloc / peer_open); with flag blocks and an epoch the launch signals the peers
        and the stream waits for theirs.  Asynchronous."""
        texel_bytes = TEXEL_BYTES.get(fmt, 16)   # an unknown format is rejected by the C ABI
        src_ptr = _device_pointer(d_level0, 6 * width * height * texel_bytes, "d_level0", self.device)
        self._after_torch()
        slots = (ctypes.c_void_p * world)(*slot_addresses)
        flags = (ctypes.c_void_p * world)(*flag_addresses) if flag_addresses is not None else None
        self._check(self._lib.datum_ibl_sh9_partial_peers(self._handle, src_ptr, fmt, width, height, row_begin, row_end, rank, world, slots, flags, epoch))

    def sh9_finish(self, partial):
        """data/project.comp:99-105 on the 28 (all-reduced) partial sums -> float32 [9][3]."""
        partial = np.ascontiguousarray(partial, dtype=np.float64)
        if partial.size != 28:
            raise ValueError("partial must hold 28 values")
        sh = np.zeros((9, 3), np.float32)
        self._lib.datum_ibl_sh9_finish(partial.ctypes.data, sh.ctypes.data)
        return sh

    def project_sh9(self, level0, fmt, width, height):
        """SH9 of a host level-0 cube (uint32 rgbe words or RGBA float32) -> float32 [9][3]."""
        texel_bytes = TEXEL_BYTES.get(fmt, 16)   # an unknown format is rejected by the C ABI
        ptr = _host_pointer(level0, 6 * width * height * texel_bytes, "level0")
        sh = np.zeros((9, 3), np.float32)
        self._check(self._lib.datum_ibl_project_sh9(self._handle, ptr, fmt, width, height, sh.ctypes.data))
        return sh

    def sh9_irradiance_cube(self, sh, width, height, want_words=True, want_f32=True):
        """Diffuse irradiance cube from SH9 (data/lighting.inc:351-366, 371)."""
        sh = np.ascontiguousarray(sh, dtype=np.float32)
        if sh.size != 27:
            raise ValueError("sh must hold 27 values")
        words = np.zeros(6 * width * height, np.uint32) if want_words else None
        f32 = np.zeros((6 * width * height, 3), np.float32) if want_f32 else None
        self._check(self._lib.datum_ibl_sh9_irradiance_cube(
            self._handle, sh.ctypes.data, width, height,
            words.ctypes.data if want_words else None, f32.ctypes.data if want_f32 else None))
        return words, f32

    # ---- 2D LUTs ----

    def image_pack_envbrdf(self, width, height, bits, samples=1024):
        """tools/ibl.h:13"""
        ptr = _host_pointer(bits, width * height * 4, "bits")
        self._check(self._lib.datum_ibl_pack_envbrdf(self._handle, width, height, samples, ptr))

    def image_pack_watercolor(self, deepcolor, shallowcolor, depthscale, fresnelcolor, fresnelbias, fresnelpower, width, height, bits):
        """tools/ibl.h:15"""
        ptr = _host_pointer(bits, width * height * 4, "bits")
        deep = np.ascontiguousarray(deepcolor, dtype=np.float32)
        shallow = np.ascontiguousarray(shallowcolor, dtype=np.float32)
        fresnel = np.ascontiguousarray(fresnelcolor, dtype=np.float32)
        if deep.size != 3 or shallow.size != 3 or fresnel.size != 3:
            raise ValueError("colours must have 3 components")
        self._check(self._lib.datum_ibl_pack_watercolor(
            self._handle, deep.ctypes.data, shallow.ctypes.data, float(depthscale), fresnel.ctypes.data,
            float(fresnelbias), float(fresnelpower), width, height, ptr))

    # ---- equirect HDR image -> cube chain: tools/ibl.cpp:283-288 ----

    def image_pack_cube_ibl(self, image, width, height, levels, bits, samples=1024):
        """tools/ibl.h:11.  `image` is an (H, W, 4) float32 array: HDRImage::bits (tools/hdr.h:24)."""
        fn = getattr(self._lib, "datum_ibl_pack_cube_ibl", None)
        if fn is None:
            raise IblError("libdatum_ibl_cuda was built without the equirect resample stage")
        image = _equirect_image(image)
        ptr = _host_pointer(bits, image_datasize(width, height, 6, levels), "bits")
        self._check(fn(self._handle, image.shape[1], image.shape[0], image.ctypes.data, width, height, levels, samples, ptr))

    def image_pack_cube(self, image, width, height, bits):
        """tools/hdr.cpp:331-359 with levels == 1 (the only use on the IBL path): resample + edge blend."""
        fn = getattr(self._lib, "datum_ibl_pack_cube", None)
        if fn is None:
            raise IblError("libdatum_ibl_cuda was built without the equirect resample stage")
        image = _equirect_image(image)
        ptr = _host_pointer(bits, width * height * 6 * 4, "bits")
        self._check(fn(self._handle, image.shape[1], image.shape[0], image.ctypes.data, width, height, ptr))


    # ---- six ARGB32 face images -> cube chain: tools/assetbuilder.cpp:416-470 ----

    def ingest_cube_argb32(self, faces, bits):
        """The per-image loop of write_skybox_asset(fout, id, paths) (assetbuilder.cpp:443-462).
        `faces` is a (6, H, W) uint32 array of QImage::Format_ARGB32 pixels (0xAARRGGBB) in the
        caller's face order; `bits` receives level 0 (6*W*H rgbe words)."""
        faces = _face_images(faces)
        height, width = faces.shape[1], faces.shape[2]
        ptr = _host_pointer(bits, width * height * 6 * 4, "bits")
        self._check(self._lib.datum_ibl_ingest_cube_argb32(self._handle, width, height, faces.ctypes.data, ptr))

    def skybox_from_argb32(self, faces, levels, bits, samples=1024):
        """assetbuilder.cpp:443-465: ingest + image_buildmips_cube_ibl, level 0 staying on the device."""
        faces = _face_images(faces)
        height, width = faces.shape[1], faces.shape[2]
        ptr = _host_pointer(bits, image_datasize(width, height, 6, levels), "bits")
        self._check(self._lib.datum_ibl_ingest_cube_argb32_ibl(self._handle, width, height, levels, samples, faces.ctypes.data, ptr))

    # ---- equirect HDR image or six ARGB32 face images -> float chain (RGBA32F / RGBA16F) ----

    def pack_cube_float(self, fmt, image, width, height, out):
        """Level 0 of a float chain from an (H, W, 4) float32 equirect image (HDRImage::bits): the resample and
        edge blend of image_pack_cube with the format's texel stored in place of rgbe (F32: the fp32 rgb, F16:
        min(x, 65504) rounded to nearest-even, alpha 1.0).  `out`: numpy array or CPU tensor of the format's
        dtype holding 6*width*height texels.  Pixel rgb must be finite and non-negative (F32: below 2^52).
        Synchronous."""
        image = _equirect_image(image)
        ptr = _float_host_buffer(fmt, out, 6 * width * height, "out")
        self._check(self._lib.datum_ibl_pack_cube_float(self._handle, fmt, image.shape[1], image.shape[0], image.ctypes.data, width, height, ptr))

    def pack_cube_float_ibl(self, fmt, image, width, height, levels, chain, samples=1024):
        """pack_cube_float followed by buildmips_cube_float, level 0 staying on the device: `chain` (host, the
        layout of buildmips_cube_float) receives every level, level 0 included.  Synchronous."""
        image = _equirect_image(image)
        ptr = _float_host_buffer(fmt, chain, float_chain_texels(width, height, levels), "chain")
        self._check(self._lib.datum_ibl_pack_cube_float_ibl(self._handle, fmt, image.shape[1], image.shape[0], image.ctypes.data, width, height, levels, samples, ptr))

    def ingest_cube_argb32_float(self, fmt, faces, out):
        """ingest_cube_argb32 with level 0 stored in the float format: per pixel the linear rgb of srgba(pixel),
        alpha 1.0, rows mirrored.  `faces` is (6, H, W) uint32; `out` holds 6*W*H texels of the format's dtype."""
        faces = _face_images(faces)
        height, width = faces.shape[1], faces.shape[2]
        ptr = _float_host_buffer(fmt, out, 6 * width * height, "out")
        self._check(self._lib.datum_ibl_ingest_cube_argb32_float(self._handle, fmt, width, height, faces.ctypes.data, ptr))

    def skybox_float_from_argb32(self, fmt, faces, levels, chain, samples=1024):
        """ingest_cube_argb32_float followed by buildmips_cube_float, level 0 staying on the device: `chain`
        receives every level.  Synchronous."""
        faces = _face_images(faces)
        height, width = faces.shape[1], faces.shape[2]
        ptr = _float_host_buffer(fmt, chain, float_chain_texels(width, height, levels), "chain")
        self._check(self._lib.datum_ibl_ingest_cube_argb32_float_ibl(self._handle, fmt, width, height, levels, samples, faces.ctypes.data, ptr))


class MultiContext:
    """Several GPUs of one node driven from this process (wraps datum_ibl_multi): the single-process
    counterpart of dist.py.  `devices` may list a device more than once."""

    def __init__(self, devices):
        self._lib = _lib.load()
        self.devices = [int(d) for d in devices]
        handle = ctypes.c_void_p()
        arr = (ctypes.c_int * len(self.devices))(*self.devices)
        if self._lib.datum_ibl_multi_create(len(self.devices), arr, ctypes.byref(handle)):
            raise IblError(self._lib.datum_ibl_last_error().decode("utf-8", "replace"))
        self._handle = handle

    def _check(self, status):
        if status:
            raise IblError(self._lib.datum_ibl_last_error().decode("utf-8", "replace"))

    def close(self):
        if getattr(self, "_handle", None):
            self._lib.datum_ibl_multi_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            if not sys.is_finalizing():
                self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def image_buildmips_cube_ibl(self, width, height, levels, bits, samples=1024):
        """tools/ibl.h:9 with ONE probe shared by the devices (rows of every big level split, NVLink peer stores)."""
        ptr = _host_pointer(bits, image_datasize(width, height, 6, levels), "bits")
        self._check(self._lib.datum_ibl_multi_buildmips_cube_ibl(self._handle, width, height, levels, samples, ptr))

    def buildmips_cube_float(self, fmt, width, height, levels, chain, samples=1024):
        """IblContext.buildmips_cube_float with ONE probe shared by the devices (rows of every big level split,
        NVLink peer stores).  Level 0 stays the caller's; the other levels equal the one-device chain's up to the
        re-cut tiles.  Synchronous."""
        if hasattr(chain, "is_cuda") and chain.is_cuda:
            raise ValueError("chain must be a host buffer")
        _check_dtype(chain, _float_dtype(fmt), "chain")
        ptr = _host_pointer(chain, float_chain_texels(width, height, levels) * _texel_bytes(fmt), "chain")
        self._check(self._lib.datum_ibl_multi_buildmips_cube_float(self._handle, fmt, width, height, levels, samples, ptr))

    def bake_probes(self, width, height, levels, payloads, samples=1024, sh9=False):
        """IblContext.bake_probes with probe p on devices[p % ndev]."""
        count = len(payloads)
        need = image_datasize(width, height, 6, levels)
        pointers = (ctypes.c_void_p * max(count, 1))()
        for i, payload in enumerate(payloads):
            pointers[i] = _host_pointer(payload, need, "payloads[%d]" % i)
        sh = np.zeros((count, 9, 3), np.float32) if sh9 else None
        self._check(self._lib.datum_ibl_multi_bake_probes(self._handle, count, width, height, levels, samples, pointers, sh.ctypes.data if sh9 and count else None))
        return sh

    def bake_probes_float(self, fmt, width, height, levels, chains, samples=1024, sh9=False):
        """IblContext.bake_probes_float with probe p on devices[p % ndev]."""
        count = len(chains)
        pointers = _float_chain_pointers(fmt, width, height, levels, chains)
        sh = np.zeros((count, 9, 3), np.float32) if sh9 else None
        self._check(self._lib.datum_ibl_multi_bake_probes_float(self._handle, fmt, count, width, height, levels, samples, pointers, sh.ctypes.data if sh9 and count else None))
        return sh

    def project_sh9(self, level0, fmt, width, height):
        """IblContext.project_sh9 with the cube's rows split over the devices."""
        texel_bytes = TEXEL_BYTES.get(fmt, 16)   # an unknown format is rejected by the C ABI
        ptr = _host_pointer(level0, 6 * width * height * texel_bytes, "level0")
        sh = np.zeros((9, 3), np.float32)
        self._check(self._lib.datum_ibl_multi_project_sh9(self._handle, ptr, fmt, width, height, sh.ctypes.data))
        return sh


_default = {}
_live = weakref.WeakSet()


@atexit.register
def _drain_all():
    # At interpreter exit only drain outstanding work.  The contexts (and their streams, which
    # torch tensors may still reference) are left for process teardown: destroying them here, or
    # from __del__ while the CUDA runtime unloads, races with torch's own shutdown.
    for ctx in list(_live):
        try:
            if ctx._handle:
                ctx.synchronize()
        except Exception:
            pass


def default_context(device=0):
    ctx = _default.get(device)
    if ctx is None:
        ctx = _default[device] = IblContext(device)
    return ctx


# ---- the reference's free functions (tools/ibl.h) on the default context ----

def image_buildmips_cube_ibl(width, height, levels, bits, samples=1024):
    default_context().image_buildmips_cube_ibl(width, height, levels, bits, samples)


def image_pack_cube_ibl(image, width, height, levels, bits, samples=1024):
    default_context().image_pack_cube_ibl(image, width, height, levels, bits, samples)


def image_pack_envbrdf(width, height, bits, samples=1024):
    default_context().image_pack_envbrdf(width, height, bits, samples)


def image_pack_watercolor(deepcolor, shallowcolor, depthscale, fresnelcolor, fresnelbias, fresnelpower, width, height, bits):
    default_context().image_pack_watercolor(deepcolor, shallowcolor, depthscale, fresnelcolor, fresnelbias, fresnelpower, width, height, bits)


def project_sh9(level0, fmt, width, height):
    return default_context().project_sh9(level0, fmt, width, height)
