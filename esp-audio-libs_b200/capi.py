"""ctypes binding of include/esp_audio_b200.h (the drop-in C ABI)."""
import ctypes as C
import os
import re

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
# (ESPB_LIBRARY: another build of the same library, e.g. a kernel variant under tools/sweep_kernel.sh)
_SO = os.environ.get("ESPB_LIBRARY") or os.path.join(_HERE, "libesp_audio_b200.so")
_HEADER = os.path.join(_ROOT, "include", "esp_audio_b200.h")

SUBSAMPLE_INTERPOLATE, BLACKMAN_HARRIS, INCLUDE_LOWPASS = 0x1, 0x2, 0x4
MODE_FAST, MODE_EXACT = 0, 1
OPT_PLAN_CACHE, OPT_KERNEL_TIMING, OPT_OVERLAP_STAGING = 1, 2, 3


class EspbError(RuntimeError):
    pass


class _Result(C.Structure):
    _fields_ = [("input_used", C.c_uint), ("output_generated", C.c_uint)]


class _Layout(C.Structure):
    _fields_ = [("stream_stride", C.c_int64), ("channel_stride", C.c_int64), ("frame_stride", C.c_int64)]


class _Coeffs(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("a0", "a1", "a2", "b1", "b2")]


class _Config(C.Structure):
    _fields_ = [("source_sample_rate", C.c_float), ("target_sample_rate", C.c_float),
                ("source_bits_per_sample", C.c_uint8), ("target_bits_per_sample", C.c_uint8),
                ("channels", C.c_uint8), ("use_pre_or_post_filter", C.c_uint8),
                ("subsample_interpolate", C.c_uint8), ("number_of_taps", C.c_uint16),
                ("number_of_filters", C.c_uint16)]


class _WResults(C.Structure):
    _fields_ = [("frames_used", C.c_size_t), ("frames_generated", C.c_size_t),
                ("predicted_frames_used", C.c_size_t), ("clipped_samples", C.c_uint64)]


_lib = None


def library_path():
    return _SO


def declared_symbols():
    """Every function name include/esp_audio_b200.h declares."""
    with open(_HEADER) as fh:
        text = fh.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(espb_\w+)\s*\(", text)))


def lib():
    """Load the product library; fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise EspbError(f"{_SO} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)")
    L = C.CDLL(_SO)
    vp, i, f, u32, u64, i64, sz = C.c_void_p, C.c_int, C.c_float, C.c_uint32, C.c_uint64, C.c_int64, C.c_size_t
    sig = {
        "espb_last_error": (C.c_char_p, []),
        "espb_abi_version": (i, []),
        "espb_device_count": (i, []),
        "espb_set_device": (i, [i]),
        "espb_device_info": (i, [C.POINTER(i), C.POINTER(i), C.POINTER(i), C.POINTER(sz), C.c_char_p, i]),
        "espb_malloc": (vp, [sz]),
        "espb_free": (None, [vp]),
        "espb_malloc_host": (vp, [sz]),
        "espb_free_host": (None, [vp]),
        "espb_memcpy_h2d": (i, [vp, vp, sz, vp]),
        "espb_memcpy_d2h": (i, [vp, vp, sz, vp]),
        "espb_memset": (i, [vp, i, sz, vp]),
        "espb_stream_create": (vp, []),
        "espb_stream_destroy": (None, [vp]),
        "espb_stream_sync": (i, [vp]),
        "espb_device_sync": (i, []),
        "espb_event_create": (vp, []),
        "espb_event_destroy": (None, [vp]),
        "espb_event_record": (i, [vp, vp]),
        "espb_event_elapsed_ms": (i, [vp, vp, C.POINTER(f)]),
        "espb_launch_count": (u64, []),
        "espb_resampleInit": (vp, [i, i, i, i, f, i]),
        "espb_resampleFree": (None, [vp]),
        "espb_resampleReset": (i, [vp, vp]),
        "espb_resampleAdvancePosition": (None, [vp, f]),
        "espb_resampleGetPosition": (f, [vp]),
        "espb_resampleGetRequiredSamples": (C.c_uint, [vp, i, f]),
        "espb_resampleGetExpectedOutput": (C.c_uint, [vp, i, f]),
        "espb_resampleSetMode": (i, [vp, i]),
        "espb_resampleSetOption": (i, [vp, i, i]),
        "espb_resampleGetKernelTime": (i, [vp, C.POINTER(f), C.POINTER(i)]),
        "espb_resampleGetFlags": (i, [vp]),
        "espb_resampleGetState": (None, [vp, C.POINTER(f), C.POINTER(i)]),
        "espb_resampleCopyFilters": (i, [vp, vp]),
        "espb_resampleProcessInterleaved": (_Result, [vp, vp, i64, i, vp, i64, i, f, vp]),
        "espb_resampleProcess": (_Result, [vp, vp, i64, i64, i, vp, i64, i64, i, f, vp]),
        "espb_resampleProcessPlanes": (_Result, [vp, vp, i, vp, i, f, vp]),
        "espb_resampleProcessLayout": (_Result, [vp, vp, C.POINTER(_Layout), i, vp, C.POINTER(_Layout), i, f, vp]),
        "espb_resampleProcessInterleavedHost": (_Result, [vp, vp, i64, i, vp, i64, i, f]),
        "espb_biquad_lowpass": (None, [C.POINTER(_Coeffs), C.c_double]),
        "espb_biquad_highpass": (None, [C.POINTER(_Coeffs), C.c_double]),
        "espb_biquad_init": (vp, [i, i, C.POINTER(_Coeffs), f]),
        "espb_biquad_free": (None, [vp]),
        "espb_biquad_reset": (i, [vp, vp]),
        "espb_biquad_apply_buffer": (i, [vp, vp, C.POINTER(_Layout), i, i, vp]),
        "espb_biquad_apply_samples": (i, [vp, vp, vp]),
        "espb_biquad_set_time_blocks": (i, [vp, i, i]),
        "espb_resampler_set_biquad_time_blocks": (i, [vp, i, i]),
        "espb_last_status": (i, []),
        "espb_resampleGroupsIsFused": (i, [vp]),
        "espb_resampleGroupsReset": (i, [vp, i, vp]),
        "espb_nccl_version": (i, []),
        "espb_measure_host_link": (i, [i, vp, sz, sz, i, C.POINTER(C.c_double)]),
        "espb_measure_host_link_pattern": (i, [i, sz, sz, i, C.POINTER(C.c_double)]),
        "espb_link_probe_create": (vp, [sz, sz]),
        "espb_link_probe_run": (i, [vp, i, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "espb_link_probe_free": (None, [vp]),
        "espb_multi_last_error": (C.c_char_p, []),
        "espb_shard_range": (None, [i64, i, i, C.POINTER(i64), C.POINTER(i64)]),
        "espb_multi_create": (vp, [i, vp]),
        "espb_multi_free": (None, [vp]),
        "espb_multi_size": (i, [vp]),
        "espb_multi_device": (i, [vp, i]),
        "espb_multi_allgather_u64": (i, [vp, vp, vp, i, vp]),
        "espb_multi_gather_words": (i, [vp, vp, i, vp]),
        "espb_dist_unique_id": (i, [vp]),
        "espb_dist_init": (vp, [vp, i, i]),
        "espb_dist_free": (None, [vp]),
        "espb_dist_rank": (i, [vp]),
        "espb_dist_world": (i, [vp]),
        "espb_dist_allgather_u64": (i, [vp, vp, i, vp]),
        "espb_dist_barrier": (i, [vp]),
        "espb_resampler_set_option": (i, [vp, i, i]),
        "espb_resampler_get_kernel_time": (i, [vp, C.POINTER(f), C.POINTER(i)]),
        "espb_biquad_block_stats": (i, [vp, C.POINTER(u64), C.POINTER(i)]),
        "espb_resampler_biquad_block_stats": (i, [vp, C.POINTER(u64), C.POINTER(i)]),
        "espb_biquad_get_state": (i, [vp, vp]),
        "espb_quantized_to_float": (i, [vp, vp, u64, C.c_uint8, f, vp]),
        "espb_float_to_quantized": (i, [vp, vp, u64, C.c_uint8, vp, vp]),
        "espb_float_to_quantized_sync": (u32, [vp, vp, u64, C.c_uint8, vp]),
        "espb_quantized_to_float_rows": (i, [vp, i64, vp, i64, i, u32, C.c_uint8, f, vp]),
        "espb_float_to_quantized_rows": (i, [vp, i64, vp, i64, i, u32, C.c_uint8, vp, vp]),
        "espb_resampler_create": (vp, [i, sz, sz, C.POINTER(_Config)]),
        "espb_resampler_free": (None, [vp]),
        "espb_resampler_set_mode": (i, [vp, i]),
        "espb_resampler_policy": (i, [vp, C.POINTER(_Coeffs), C.POINTER(f), C.POINTER(f), C.POINTER(i)]),
        "espb_resampler_resample": (_WResults, [vp, vp, i64, vp, i64, sz, sz, f, vp, vp]),
        "espb_resampler_resample_host": (_WResults, [vp, vp, i64, vp, i64, sz, sz, f, vp]),
        "espb_resampler_resample_async": (_WResults, [vp, vp, i64, vp, i64, sz, sz, f, vp]),
        "espb_resampler_clipped_dev": (vp, [vp]),
        "espb_plan_filter_bank": (i, [i, i, f, i, vp, C.POINTER(i)]),
        "espb_plan_schedule": (i, [i, i, i, f, i, i, i, f, C.POINTER(C.c_uint), C.POINTER(C.c_uint), C.POINTER(f),
                                   C.POINTER(i), vp, vp, vp, vp]),
        "espb_plan_schedule_segments": (i, [i, i, i, f, i, i, i, f, C.POINTER(C.c_uint), C.POINTER(C.c_uint),
                                            C.POINTER(f), C.POINTER(i), vp, vp, vp, vp]),
        "espb_plan_passes": (i, [i, i, i, f, i, i, i, f, i, i, vp, vp, i, vp, i]),
        "espb_plan_policy": (i, [C.POINTER(_Config), C.POINTER(_Coeffs), C.POINTER(f), C.POINTER(f), C.POINTER(i)]),
        "espb_checksum_u32": (i, [vp, u64, vp, vp]),
        "espb_resampleGroupsInit": (vp, [i, C.POINTER(i), i, i, i, f, i]),
        "espb_resampleGroupsFree": (None, [vp]),
        "espb_resampleGroupsCount": (i, [vp]),
        "espb_resampleGroupsFirstStream": (i, [vp, i]),
        "espb_resampleGroupsContext": (vp, [vp, i]),
        "espb_resampleGroupsSetMode": (i, [vp, i]),
        "espb_resampleGroupsProcessInterleaved": (i, [vp, vp, i64, C.POINTER(i), vp, i64, C.POINTER(i), C.POINTER(f),
                                                      C.POINTER(_Result), vp]),
        "espb_wav_decoder_create": (vp, []),
        "espb_wav_decoder_free": (None, [vp]),
        "espb_wav_decoder_decode_header": (i, [vp, vp, sz]),
        "espb_wav_decoder_next": (i, [vp, vp]),
        "espb_wav_decoder_reset": (None, [vp]),
        "espb_wav_decoder_state": (i, [vp]),
        "espb_wav_decoder_bytes_processed": (sz, [vp]),
        "espb_wav_decoder_bytes_to_skip": (sz, [vp]),
        "espb_wav_decoder_bytes_needed": (sz, [vp]),
        "espb_wav_decoder_chunk_name": (vp, [vp]),  # 4 raw bytes (may hold NULs)
        "espb_wav_decoder_chunk_bytes_left": (sz, [vp]),
        "espb_wav_decoder_sample_rate": (u32, [vp]),
        "espb_wav_decoder_num_channels": (C.c_uint16, [vp]),
        "espb_wav_decoder_bits_per_sample": (C.c_uint16, [vp]),
        "espb_wav_write_header": (sz, [vp, u32, C.c_uint16, C.c_uint16, u32]),
        "espb_dsps_add_s16": (i, [vp, vp, vp, i64, i, i, i, i, vp]),
        "espb_dsps_mulc_s16": (i, [vp, vp, i64, C.c_int16, i, i, vp]),
        "espb_measure_fp32_fma_peak": (i, [C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "espb_measure_fp32_fma_peak2": (i, [C.POINTER(C.c_double), C.POINTER(C.c_double)]),
        "espb_measure_fp32_tile_pattern": (i, [C.POINTER(C.c_double)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def _err():
    return lib().espb_last_error().decode(errors="replace")


def _check(rc, what):
    if rc != 0:
        raise EspbError(f"{what} failed ({rc}): {_err()}")


def device_count():
    return lib().espb_device_count()


def set_device(d):
    _check(lib().espb_set_device(d), "espb_set_device")


def device_info():
    sm, ma, mi, mem = C.c_int(0), C.c_int(0), C.c_int(0), C.c_size_t(0)
    name = C.create_string_buffer(256)
    _check(lib().espb_device_info(C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem), name, 256), "device_info")
    return dict(sm_count=sm.value, cc=(ma.value, mi.value), total_mem=mem.value, name=name.value.decode())


def launch_count():
    return int(lib().espb_launch_count())


def measure_fp32_fma_peak():
    tf, mhz = C.c_double(0), C.c_double(0)
    _check(lib().espb_measure_fp32_fma_peak(C.byref(tf), C.byref(mhz)), "measure_fp32_fma_peak")
    return tf.value, mhz.value


def plan_filter_bank(taps, filters, lowpass, flags):
    """Host-only: (bank (filters+1, taps) float32, effective flags) or None for invalid parameters."""
    bank = np.zeros((max(filters, 0) + 1, max(taps, 1)), np.float32)
    eff = C.c_int(0)
    if lib().espb_plan_filter_bank(taps, filters, lowpass, flags, bank.ctypes.data, C.byref(eff)) != 0:
        return None
    return bank, int(eff.value)


def plan_schedule(taps, filters, flags, offset, index, n_in, n_out, ratio, want_entries=True):
    """Host-only dry run of the position state machine."""
    used, gen, eo, ei = C.c_uint(0), C.c_uint(0), C.c_float(0), C.c_int(0)
    n = max(n_out, 1)
    ws, ph, w, kind = (np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.int32))
    ptrs = [a.ctypes.data if want_entries else None for a in (ws, ph, w, kind)]
    _check(lib().espb_plan_schedule(taps, filters, flags, offset, index, n_in, n_out, ratio, C.byref(used),
                                    C.byref(gen), C.byref(eo), C.byref(ei), *ptrs), "plan_schedule")
    g = int(gen.value)
    return dict(used=int(used.value), generated=g, end_offset=np.float32(eo.value), end_index=int(ei.value),
                ws=ws[:g], phase=ph[:g], w=w[:g], kind=kind[:g])


def plan_schedule_segments(taps, filters, flags, offset, index, n_in, n_out, ratio, want_entries=True):
    """The same dry run through the closed-form (segmented) planner of the processing path; adds `segments`."""
    used, gen, eo, ei = C.c_uint(0), C.c_uint(0), C.c_float(0), C.c_int(0)
    n = max(n_out, 1)
    ws, ph, w, kind = (np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.int32))
    ptrs = [a.ctypes.data if want_entries else None for a in (ws, ph, w, kind)]
    rc = lib().espb_plan_schedule_segments(taps, filters, flags, offset, index, n_in, n_out, ratio, C.byref(used),
                                           C.byref(gen), C.byref(eo), C.byref(ei), *ptrs)
    if rc < 0:
        _check(rc, "plan_schedule_segments")
    g = int(gen.value)
    return dict(used=int(used.value), generated=g, end_offset=np.float32(eo.value), end_index=int(ei.value),
                ws=ws[:g], phase=ph[:g], w=w[:g], kind=kind[:g], segments=int(rc))


def plan_passes(taps, filters, flags, offset, index, n_in, n_out, ratio, blocks_per_pass=4, chunk_rows=32):
    """Host-only: the chunk table of a call: (chunk_start, chunk_pass, pass_chunk_begin) int32 arrays."""
    n = lib().espb_plan_passes(taps, filters, flags, offset, index, n_in, n_out, ratio, blocks_per_pass, chunk_rows,
                               None, None, 0, None, 0)
    if n < 0:
        raise EspbError(f"plan_passes: {_err()}")
    cs, cp = np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.int32)
    pcb = np.zeros(max(n, 1) + 2, np.int32)
    lib().espb_plan_passes(taps, filters, flags, offset, index, n_in, n_out, ratio, blocks_per_pass, chunk_rows,
                           cs.ctypes.data, cp.ctypes.data, n, pcb.ctypes.data, pcb.size)
    n_passes = int(cp[n - 1]) + 1 if n else 0
    return cs[:n], cp[:n], pcb[: n_passes + 1]


def plan_policy(src_rate, dst_rate, src_bits, dst_bits, channels, use_filter, interpolate, taps, filters):
    cfg = _Config(float(src_rate), float(dst_rate), src_bits, dst_bits, channels, int(use_filter), int(interpolate),
                  taps, filters)
    c, ratio, lp, flags = _Coeffs(), C.c_float(0), C.c_float(0), C.c_int(0)
    kind = lib().espb_plan_policy(C.byref(cfg), C.byref(c), C.byref(ratio), C.byref(lp), C.byref(flags))
    return dict(filter={0: "none", 1: "pre", 2: "post"}[kind],
                coeffs=np.array([c.a0, c.a1, c.a2, c.b1, c.b2], np.float32), sample_ratio=np.float32(ratio.value),
                art_lowpass=np.float32(lp.value), art_flags=int(flags.value))


def measure_host_link(devices=None, nbytes=1 << 30, slab_bytes=64 << 20, reps=3):
    """Aggregate GB/s per direction of pinned cudaMemcpyAsync on `devices` (None: the current one), all at once."""
    out = (C.c_double * 6)()
    if devices is None:
        rc = lib().espb_measure_host_link(0, None, nbytes, slab_bytes, reps, out)
    else:
        arr = (C.c_int * len(devices))(*devices)
        rc = lib().espb_measure_host_link(len(devices), arr, nbytes, slab_bytes, reps, out)
    _check(rc, "measure_host_link")
    return dict(h2d_gbs=out[0], d2h_gbs=out[1], duplex_each_gbs=out[2], duplex_sum_gbs=out[4], duplex_seconds=out[5],
                bytes_per_direction_per_device=nbytes, slab_bytes=slab_bytes)


def measure_host_link_pattern(pattern, nbytes=1 << 30, slab_bytes=64 << 20, reps=2):
    """GB/s per direction of one pattern (0 H2D, 1 D2H, 2 both) on the current device."""
    v = C.c_double(0)
    _check(lib().espb_measure_host_link_pattern(pattern, nbytes, slab_bytes, reps, C.byref(v)), "measure_host_link")
    return float(v.value)


def measure_fp32_tile_pattern():
    tf = C.c_double(0)
    _check(lib().espb_measure_fp32_tile_pattern(C.byref(tf)), "measure_fp32_tile_pattern")
    return tf.value


def measure_fp32_fma_peak2():
    a, b = C.c_double(0), C.c_double(0)
    _check(lib().espb_measure_fp32_fma_peak2(C.byref(a), C.byref(b)), "measure_fp32_fma_peak2")
    return a.value, b.value


class DeviceBuffer:
    """Device memory through espb_malloc / espb_free / espb_memcpy_*."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        self.ptr = lib().espb_malloc(max(self.nbytes, 1))
        if not self.ptr:
            raise EspbError(f"espb_malloc({nbytes}) failed: {_err()}")

    @classmethod
    def from_numpy(cls, a, stream=None):
        a = np.ascontiguousarray(a)
        b = cls(a.nbytes)
        b.upload(a, stream)
        return b

    def upload(self, a, stream=None):
        a = np.ascontiguousarray(a)
        assert a.nbytes <= self.nbytes
        if a.nbytes:
            _check(lib().espb_memcpy_h2d(self.ptr, a.ctypes.data, a.nbytes, stream), "h2d")
            _check(lib().espb_stream_sync(stream), "sync")  # pageable source: keep it simple and safe

    def download(self, dtype, count=None, stream=None):
        dtype = np.dtype(dtype)
        if count is None:
            count = self.nbytes // dtype.itemsize
        out = np.empty(count, dtype)
        if out.nbytes:
            _check(lib().espb_memcpy_d2h(out.ctypes.data, self.ptr, out.nbytes, stream), "d2h")
            _check(lib().espb_stream_sync(stream), "sync")
        return out

    def zero(self, stream=None):
        _check(lib().espb_memset(self.ptr, 0, self.nbytes, stream), "memset")

    def free(self):
        if getattr(self, "ptr", None):
            lib().espb_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedBuffer:
    """Page-locked host memory exposed as a numpy array."""

    def __init__(self, count, dtype):
        self.dtype = np.dtype(dtype)
        self.nbytes = int(count) * self.dtype.itemsize
        self.ptr = lib().espb_malloc_host(max(self.nbytes, 1))
        if not self.ptr:
            raise EspbError(f"espb_malloc_host failed: {_err()}")
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(count))

    def free(self):
        if getattr(self, "ptr", None):
            self.array = None
            lib().espb_free_host(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class ResampleBatch:
    """`num_streams` reference contexts (art_resampler.h) sharing one configuration."""

    def __init__(self, num_streams, channels, taps, filters, lowpass_ratio, flags, mode=MODE_FAST):
        self.h = lib().espb_resampleInit(num_streams, channels, taps, filters, lowpass_ratio, flags)
        if not self.h:
            raise EspbError(f"espb_resampleInit returned NULL: {_err()}")
        self.num_streams, self.channels, self.taps, self.filters = num_streams, channels, taps, filters
        self.set_mode(mode)

    def free(self):
        if getattr(self, "h", None):
            lib().espb_resampleFree(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def set_mode(self, mode):
        _check(lib().espb_resampleSetMode(self.h, mode), "resampleSetMode")

    def reset(self, stream=None):
        _check(lib().espb_resampleReset(self.h, stream), "resampleReset")

    def set_option(self, option, value):
        _check(lib().espb_resampleSetOption(self.h, option, value), "resampleSetOption")

    def kernel_time(self):
        ms, n = C.c_float(0), C.c_int(0)
        _check(lib().espb_resampleGetKernelTime(self.h, C.byref(ms), C.byref(n)), "resampleGetKernelTime")
        return float(ms.value), int(n.value)

    def advance(self, delta):
        lib().espb_resampleAdvancePosition(self.h, delta)

    def position(self):
        return float(lib().espb_resampleGetPosition(self.h))

    def required(self, n_out, ratio):
        return int(lib().espb_resampleGetRequiredSamples(self.h, n_out, ratio))

    def expected(self, n_in, ratio):
        return int(lib().espb_resampleGetExpectedOutput(self.h, n_in, ratio))

    def flags(self):
        return int(lib().espb_resampleGetFlags(self.h))

    def state(self):
        off, idx = C.c_float(0), C.c_int(0)
        lib().espb_resampleGetState(self.h, C.byref(off), C.byref(idx))
        return np.float32(off.value), int(idx.value)

    def bank(self):
        out = np.empty((self.filters + 1, self.taps), np.float32)
        _check(lib().espb_resampleCopyFilters(self.h, out.ctypes.data), "resampleCopyFilters")
        return out

    # ---- device-pointer calls (what a C caller does) ----
    def process_interleaved_dev(self, d_in, in_stride, n_in, d_out, out_stride, n_out, ratio, stream=None):
        r = lib().espb_resampleProcessInterleaved(self.h, d_in, in_stride, n_in, d_out, out_stride, n_out, ratio,
                                                  stream)
        if r.input_used == 0 and r.output_generated == 0 and _err():
            raise EspbError(f"espb_resampleProcessInterleaved: {_err()}")
        return int(r.input_used), int(r.output_generated)

    def process_interleaved_host(self, h_in_ptr, in_stride, n_in, h_out_ptr, out_stride, n_out, ratio):
        r = lib().espb_resampleProcessInterleavedHost(self.h, h_in_ptr, in_stride, n_in, h_out_ptr, out_stride,
                                                      n_out, ratio)
        if r.input_used == 0 and r.output_generated == 0 and _err():
            raise EspbError(f"espb_resampleProcessInterleavedHost: {_err()}")
        return int(r.input_used), int(r.output_generated)

    # ---- numpy convenience (tests) ----
    def process_interleaved(self, x, n_out, ratio, n_in=None):
        """x: (num_streams, n_in*channels) float32.  Returns (y (num_streams, gen*channels), used, generated)."""
        x = np.ascontiguousarray(x, np.float32)
        x = x.reshape(self.num_streams, x.size // self.num_streams)
        row = x.shape[1]
        if n_in is None:
            n_in = row // self.channels
        d_in = DeviceBuffer.from_numpy(x if x.size else np.zeros(1, np.float32))
        out_row = max(n_out, 1) * self.channels
        d_out = DeviceBuffer(self.num_streams * out_row * 4)
        d_out.zero()
        used, gen = self.process_interleaved_dev(d_in.ptr, row, n_in, d_out.ptr, out_row, n_out, ratio)
        y = d_out.download(np.float32).reshape(self.num_streams, out_row)[:, : gen * self.channels].copy()
        d_in.free()
        d_out.free()
        return y, used, gen

    def process_planar(self, x, n_out, ratio):
        """x: (num_streams, channels, n_in) float32 -> (y (num_streams, channels, gen), used, generated)."""
        x = np.ascontiguousarray(x, np.float32)
        ns, ch, n_in = x.shape
        d_in = DeviceBuffer.from_numpy(x)
        cap = max(n_out, 1)
        d_out = DeviceBuffer(ns * ch * cap * 4)
        d_out.zero()
        r = lib().espb_resampleProcess(self.h, d_in.ptr, ch * n_in, n_in, n_in, d_out.ptr, ch * cap, cap, n_out,
                                       ratio, None)
        y = d_out.download(np.float32).reshape(ns, ch, cap)[:, :, : r.output_generated].copy()
        d_in.free()
        d_out.free()
        return y, int(r.input_used), int(r.output_generated)


    def process_planes(self, planes, n_out, ratio):
        """planes: list of num_streams*channels 1-D float32 arrays (one separately allocated device buffer each,
        plane q = stream q // channels, channel q % channels) -> (list of output planes, used, generated)."""
        n = len(planes)
        n_in = len(planes[0])
        cap = max(n_out, 1)
        d_in = [DeviceBuffer.from_numpy(np.ascontiguousarray(p, np.float32) if n_in else np.zeros(1, np.float32))
                for p in planes]
        d_out = [DeviceBuffer(cap * 4) for _ in range(n)]
        for d in d_out:
            d.zero()
        pin = (C.c_void_p * n)(*[d.ptr for d in d_in])
        pout = (C.c_void_p * n)(*[d.ptr for d in d_out])
        r = lib().espb_resampleProcessPlanes(self.h, pin, n_in, pout, n_out, ratio, None)
        if _err():
            raise EspbError(f"espb_resampleProcessPlanes: {_err()}")
        ys = [d.download(np.float32)[: r.output_generated].copy() for d in d_out]
        for d in d_in + d_out:
            d.free()
        return ys, int(r.input_used), int(r.output_generated)


class ResampleGroups:
    """Ratio groups (ASRC): one batch context per group of streams that share a clock."""

    def __init__(self, streams_per_group, channels, taps, filters, lowpass_ratio, flags, mode=MODE_FAST):
        self.sizes = [int(v) for v in streams_per_group]
        arr = (C.c_int * len(self.sizes))(*self.sizes)
        self.h = lib().espb_resampleGroupsInit(len(self.sizes), arr, channels, taps, filters, lowpass_ratio, flags)
        if not self.h:
            raise EspbError(f"espb_resampleGroupsInit returned NULL: {_err()}")
        self.channels, self.num_streams = channels, sum(self.sizes)
        _check(lib().espb_resampleGroupsSetMode(self.h, mode), "resampleGroupsSetMode")

    def context(self, k):
        return lib().espb_resampleGroupsContext(self.h, k)

    def is_fused(self):
        return bool(lib().espb_resampleGroupsIsFused(self.h))

    def reset(self, k, stream=None):
        _check(lib().espb_resampleGroupsReset(self.h, k, stream), "resampleGroupsReset")

    def advance(self, k, delta):
        lib().espb_resampleAdvancePosition(self.context(k), delta)

    def state(self, k):
        off, idx = C.c_float(0), C.c_int(0)
        lib().espb_resampleGetState(self.context(k), C.byref(off), C.byref(idx))
        return np.float32(off.value), int(idx.value)

    def process_interleaved(self, x, n_in, n_out, ratios):
        """x: (num_streams, row) float32 with row >= max(n_in)*channels; n_in / n_out / ratios: one entry per
        group.  Returns (y (num_streams, max(n_out)*channels), [(used, generated)] per group)."""
        x = np.ascontiguousarray(x, np.float32)
        row = x.shape[1]
        out_row = max(max(n_out), 1) * self.channels
        d_in = DeviceBuffer.from_numpy(x if x.size else np.zeros(1, np.float32))
        d_out = DeviceBuffer(self.num_streams * out_row * 4)
        d_out.zero()
        k = len(self.sizes)
        res = (_Result * k)()
        _check(lib().espb_resampleGroupsProcessInterleaved(
            self.h, d_in.ptr, row, (C.c_int * k)(*[int(v) for v in n_in]), d_out.ptr, out_row,
            (C.c_int * k)(*[int(v) for v in n_out]), (C.c_float * k)(*[float(v) for v in ratios]), res, None),
            "resampleGroupsProcessInterleaved")
        y = d_out.download(np.float32).reshape(self.num_streams, out_row)
        d_in.free()
        d_out.free()
        return y, [(int(r.input_used), int(r.output_generated)) for r in res]

    def free(self):
        if getattr(self, "h", None):
            lib().espb_resampleGroupsFree(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def biquad_lowpass(frequency):
    c = _Coeffs()
    lib().espb_biquad_lowpass(C.byref(c), frequency)
    return np.array([c.a0, c.a1, c.a2, c.b1, c.b2], np.float32)


def biquad_highpass(frequency):
    c = _Coeffs()
    lib().espb_biquad_highpass(C.byref(c), frequency)
    return np.array([c.a0, c.a1, c.a2, c.b1, c.b2], np.float32)


class BiquadBatch:
    def __init__(self, num_series, num_sections, coeffs, gain=1.0):
        c = _Coeffs(*[float(v) for v in coeffs])
        self.h = lib().espb_biquad_init(num_series, num_sections, C.byref(c), gain)
        if not self.h:
            raise EspbError(f"espb_biquad_init returned NULL: {_err()}")
        self.num_series, self.num_sections = num_series, num_sections

    def free(self):
        if getattr(self, "h", None):
            lib().espb_biquad_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def reset(self, stream=None):
        _check(lib().espb_biquad_reset(self.h, stream), "biquad_reset")

    def set_time_blocks(self, block_rows, warmup_rows):
        _check(lib().espb_biquad_set_time_blocks(self.h, block_rows, warmup_rows), "biquad_set_time_blocks")

    def block_stats(self):
        """(blocks repaired so far, current warm-up rows) of the time-block mode."""
        n, w = C.c_uint64(0), C.c_int(0)
        _check(lib().espb_biquad_block_stats(self.h, C.byref(n), C.byref(w)), "biquad_block_stats")
        return int(n.value), int(w.value)

    def apply_dev(self, d_buf, layout, channels, n_samples, stream=None):
        lay = _Layout(*layout)
        _check(lib().espb_biquad_apply_buffer(self.h, d_buf, C.byref(lay), channels, n_samples, stream),
               "biquad_apply_buffer")

    def apply_samples(self, x):
        """One sample per series (biquad_apply_sample for the whole bank); returns the filtered samples."""
        x = np.ascontiguousarray(x, np.float32)
        d = DeviceBuffer.from_numpy(x)
        _check(lib().espb_biquad_apply_samples(self.h, d.ptr, None), "biquad_apply_samples")
        y = d.download(np.float32, x.size)
        d.free()
        return y

    def apply_interleaved(self, x, channels):
        """x: (num_streams, n*channels) float32, filtered in place on the device; returns the result."""
        x = np.ascontiguousarray(x, np.float32)
        ns, row = x.shape
        d = DeviceBuffer.from_numpy(x)
        self.apply_dev(d.ptr, (row, 1, channels), channels, row // channels)
        y = d.download(np.float32).reshape(ns, row)
        d.free()
        return y

    def state(self):
        out = np.empty((self.num_series, self.num_sections, 4), np.float32)
        _check(lib().espb_biquad_get_state(self.h, out.ctypes.data), "biquad_get_state")
        return out


def quantized_to_float(data, n, bits, gain_db=0.0):
    """numpy convenience over espb_quantized_to_float: bytes -> float32[n]."""
    data = np.ascontiguousarray(data, np.uint8)
    d_in = DeviceBuffer.from_numpy(data if data.size else np.zeros(4, np.uint8))
    d_out = DeviceBuffer(max(n, 1) * 4)
    _check(lib().espb_quantized_to_float(d_in.ptr, d_out.ptr, n, bits, gain_db, None), "quantized_to_float")
    out = d_out.download(np.float32, n)
    d_in.free()
    d_out.free()
    return out


def float_to_quantized(x, bits):
    """numpy convenience over espb_float_to_quantized_sync: float32 -> (bytes, clipped)."""
    x = np.ascontiguousarray(x, np.float32)
    nb = (bits + 7) // 8
    d_in = DeviceBuffer.from_numpy(x if x.size else np.zeros(1, np.float32))
    d_out = DeviceBuffer(max(x.size * nb, 4))
    clipped = lib().espb_float_to_quantized_sync(d_in.ptr, d_out.ptr, x.size, bits, None)
    if _err() and clipped == 0 and x.size and lib().espb_device_count() <= 0:
        raise EspbError(_err())
    out = d_out.download(np.uint8, x.size * nb)
    d_in.free()
    d_out.free()
    return out, int(clipped)


def dsps_add_s16(a, b, n, step1=1, step2=1, step_out=1, shift=0, out_init=None):
    """numpy convenience over espb_dsps_add_s16: (out int16[max(n*step_out,1)], rc).  Elements of `out` the call does
    not write keep `out_init` (default zeros), as a caller-owned buffer would."""
    a, b = np.ascontiguousarray(a, np.int16), np.ascontiguousarray(b, np.int16)
    out = np.zeros(max(n * step_out, 1), np.int16) if out_init is None else np.ascontiguousarray(out_init, np.int16)
    d_a, d_b, d_o = (DeviceBuffer.from_numpy(x if x.size else np.zeros(1, np.int16)) for x in (a, b, out))
    rc = lib().espb_dsps_add_s16(d_a.ptr, d_b.ptr, d_o.ptr, n, step1, step2, step_out, shift, None)
    res = d_o.download(np.int16, out.size)
    for d in (d_a, d_b, d_o):
        d.free()
    return res, rc


def dsps_mulc_s16(a, n, c, step_in=1, step_out=1, out_init=None):
    """numpy convenience over espb_dsps_mulc_s16: (out int16[max(n*step_out,1)], rc)."""
    a = np.ascontiguousarray(a, np.int16)
    out = np.zeros(max(n * step_out, 1), np.int16) if out_init is None else np.ascontiguousarray(out_init, np.int16)
    d_a, d_o = (DeviceBuffer.from_numpy(x if x.size else np.zeros(1, np.int16)) for x in (a, out))
    rc = lib().espb_dsps_mulc_s16(d_a.ptr, d_o.ptr, n, c, step_in, step_out, None)
    res = d_o.download(np.int16, out.size)
    d_a.free()
    d_o.free()
    return res, rc


class WavDecoder:
    """include/wav_decoder.h:54-89 over the C ABI (host only; works without a GPU)."""

    def __init__(self):
        self.h = lib().espb_wav_decoder_create()
        if not self.h:
            raise EspbError("espb_wav_decoder_create failed")

    def decode_header(self, data):
        buf = np.frombuffer(bytes(data), np.uint8) if len(data) else np.zeros(1, np.uint8)
        return lib().espb_wav_decoder_decode_header(self.h, buf.ctypes.data, len(data))

    def next(self, data):
        buf = np.frombuffer(bytes(data) + b"\0" * 16, np.uint8)
        return lib().espb_wav_decoder_next(self.h, buf.ctypes.data)

    def reset(self):
        lib().espb_wav_decoder_reset(self.h)

    def snapshot(self):
        L = lib()
        return (L.espb_wav_decoder_state(self.h), L.espb_wav_decoder_bytes_processed(self.h),
                L.espb_wav_decoder_bytes_needed(self.h), L.espb_wav_decoder_bytes_to_skip(self.h),
                L.espb_wav_decoder_chunk_bytes_left(self.h), L.espb_wav_decoder_sample_rate(self.h),
                L.espb_wav_decoder_num_channels(self.h), L.espb_wav_decoder_bits_per_sample(self.h),
                C.string_at(L.espb_wav_decoder_chunk_name(self.h), 4))

    def free(self):
        if getattr(self, "h", None):
            lib().espb_wav_decoder_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def wav_write_header(sample_rate, channels, bits, data_bytes):
    out = np.zeros(44, np.uint8)
    n = lib().espb_wav_write_header(out.ctypes.data, sample_rate, channels, bits, data_bytes)
    return out[:n].tobytes()


class _Q15Backend:
    """Same call shape as the test oracle's Q15 helpers (tests run golden cases through either)."""
    add_s16 = staticmethod(lambda a, b, n, s1=1, s2=1, so=1, shift=0: dsps_add_s16(a, b, n, s1, s2, so, shift))
    mulc_s16 = staticmethod(lambda a, n, c, si=1, so=1: dsps_mulc_s16(a, n, c, si, so))


def checksum_u32(d_ptr, num_words, stream=None):
    acc = DeviceBuffer(8)
    acc.zero(stream)
    _check(lib().espb_checksum_u32(d_ptr, num_words, acc.ptr, stream), "checksum_u32")
    v = int(acc.download(np.uint64, 1, stream)[0])
    acc.free()
    return v


class Resampler:
    """resampler::Resampler (include/resampler.h) for `num_streams` streams."""

    def __init__(self, num_streams, input_buffer_samples, output_buffer_samples, src_rate, dst_rate, src_bits,
                 dst_bits, channels, use_filter=True, interpolate=True, taps=256, filters=256, mode=MODE_FAST):
        cfg = _Config(float(src_rate), float(dst_rate), src_bits, dst_bits, channels, int(use_filter),
                      int(interpolate), taps, filters)
        self.h = lib().espb_resampler_create(num_streams, input_buffer_samples, output_buffer_samples, C.byref(cfg))
        if not self.h:
            raise EspbError(f"espb_resampler_create returned NULL: {_err()}")
        self.num_streams, self.channels = num_streams, channels
        self.src_bytes, self.dst_bytes = (src_bits + 7) // 8, (dst_bits + 7) // 8
        _check(lib().espb_resampler_set_mode(self.h, mode), "resampler_set_mode")

    def free(self):
        if getattr(self, "h", None):
            lib().espb_resampler_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def set_biquad_time_blocks(self, block_rows, warmup_rows):
        _check(lib().espb_resampler_set_biquad_time_blocks(self.h, block_rows, warmup_rows),
               "resampler_set_biquad_time_blocks")

    def set_option(self, option, value):
        _check(lib().espb_resampler_set_option(self.h, option, value), "resampler_set_option")

    def kernel_time(self):
        ms, n = C.c_float(0), C.c_int(0)
        _check(lib().espb_resampler_get_kernel_time(self.h, C.byref(ms), C.byref(n)), "resampler_get_kernel_time")
        return float(ms.value), int(n.value)

    def biquad_block_stats(self):
        n, w = C.c_uint64(0), C.c_int(0)
        _check(lib().espb_resampler_biquad_block_stats(self.h, C.byref(n), C.byref(w)), "resampler_biquad_block_stats")
        return int(n.value), int(w.value)

    def policy(self):
        c, ratio, lp, flags = _Coeffs(), C.c_float(0), C.c_float(0), C.c_int(0)
        kind = lib().espb_resampler_policy(self.h, C.byref(c), C.byref(ratio), C.byref(lp), C.byref(flags))
        return dict(filter={0: "none", 1: "pre", 2: "post"}[kind],
                    coeffs=np.array([c.a0, c.a1, c.a2, c.b1, c.b2], np.float32),
                    sample_ratio=np.float32(ratio.value), art_lowpass=np.float32(lp.value),
                    art_flags=int(flags.value))

    @staticmethod
    def _results(r, per_stream):
        return dict(frames_used=int(r.frames_used), frames_generated=int(r.frames_generated),
                    predicted_frames_used=int(r.predicted_frames_used), clipped_samples=int(r.clipped_samples),
                    clipped_per_stream=per_stream)

    def resample_dev(self, d_in, in_stride_bytes, d_out, out_stride_bytes, in_frames, out_free, gain_db=0.0,
                     stream=None):
        per = np.zeros(self.num_streams, np.uint32)
        r = lib().espb_resampler_resample(self.h, d_in, in_stride_bytes, d_out, out_stride_bytes, in_frames, out_free,
                                          gain_db, per.ctypes.data, stream)
        if _err():
            raise EspbError(f"espb_resampler_resample: {_err()}")
        return self._results(r, per)

    def resample_dev_async(self, d_in, in_stride_bytes, d_out, out_stride_bytes, in_frames, out_free, gain_db=0.0,
                           stream=None):
        """Enqueue only; clip counts stay on the device (clipped_dev())."""
        r = lib().espb_resampler_resample_async(self.h, d_in, in_stride_bytes, d_out, out_stride_bytes, in_frames,
                                                out_free, gain_db, stream)
        if _err():
            raise EspbError(f"espb_resampler_resample_async: {_err()}")
        return self._results(r, None)

    def clipped_dev(self):
        return lib().espb_resampler_clipped_dev(self.h)

    def resample_host_ptr(self, h_in, in_stride_bytes, h_out, out_stride_bytes, in_frames, out_free, gain_db=0.0):
        per = np.zeros(self.num_streams, np.uint32)
        r = lib().espb_resampler_resample_host(self.h, h_in, in_stride_bytes, h_out, out_stride_bytes, in_frames,
                                               out_free, gain_db, per.ctypes.data)
        if _err():
            raise EspbError(f"espb_resampler_resample_host: {_err()}")
        return self._results(r, per)

    def resample(self, data, in_frames, out_free, gain_db=0.0, host_path=False):
        """data: (num_streams, row_bytes) uint8.  Returns (out (num_streams, gen*ch*dst_bytes), results)."""
        data = np.ascontiguousarray(data, np.uint8)
        data = data.reshape(self.num_streams, data.size // self.num_streams)
        in_row = data.shape[1]
        out_row = (max(out_free, 1) * self.channels * self.dst_bytes + 15) & ~15
        if host_path:
            out = np.zeros((self.num_streams, out_row), np.uint8)
            src = data if data.size else np.zeros((self.num_streams, 1), np.uint8)
            res = self.resample_host_ptr(src.ctypes.data, in_row, out.ctypes.data, out_row, in_frames, out_free,
                                         gain_db)
        else:
            d_in = DeviceBuffer.from_numpy(data if data.size else np.zeros(16, np.uint8))
            d_out = DeviceBuffer(self.num_streams * out_row)
            d_out.zero()
            res = self.resample_dev(d_in.ptr, in_row, d_out.ptr, out_row, in_frames, out_free, gain_db)
            out = d_out.download(np.uint8).reshape(self.num_streams, out_row)
            d_in.free()
            d_out.free()
        n = res["frames_generated"] * self.channels * self.dst_bytes
        return out[:, :n].copy(), res
