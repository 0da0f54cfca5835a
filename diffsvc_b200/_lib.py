"""ctypes binding of libdsvc.so (include/dsvc.h) + the in-tree nvcc build.

The product path has NO CPU fallback: if the library cannot be loaded, or no sm_100 device is
visible, every compute entry point raises.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libdsvc.so")
SOURCES = ["api.cu", "diffnet.cu", "nsf.cu", "mel.cu", "pe.cu"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared"]

DSVC_MATH_TC3F16, DSVC_MATH_FP32, DSVC_MATH_TC1F16 = 0, 1, 2
MAX_STAGES = MAX_KERNELS = MAX_DILATIONS = 8


class DsvcError(RuntimeError):
    pass


def _stale():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(_HERE, "..", "include", "dsvc.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def header_crc():
    """CRC-32 of include/dsvc.h: compiled into the library (dsvc_abi()) and checked at load -- the struct layouts and
    argtypes below are mirrored by hand, a library built from another header must not be called through them."""
    import zlib
    with open(os.path.join(_HERE, "..", "include", "dsvc.h"), "rb") as f:
        return zlib.crc32(f.read()) & 0xFFFFFFFF


def build(force=False, verbose=False, extra_flags=(), out=None):
    """Compile csrc/*.cu for sm_100a into diffsvc_b200/lib/libdsvc.so (nvcc cross-compiles without a GPU).
    `extra_flags` / `out`: developer variants (e.g. -DDSVC_TIMELINE) next to the product library, loaded via DSVC_LIB."""
    if out is None:
        out = LIB_PATH
        if not force and not _stale():
            return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    tmp = out + ".tmp.%d" % os.getpid()
    # one nvcc per translation unit, in parallel (they share no device symbols), then one link
    objs, procs = [], []
    for src in SOURCES:
        obj = "%s.%s.o" % (tmp, src[:-3])
        cmd = [nvcc] + [f for f in NVCC_FLAGS if f != "-shared"] + ["-DDSVC_ABI_HASH=0x%08xu" % header_crc()] + list(extra_flags) \
            + ["-c", "-o", obj, os.path.join(CSRC, src)]
        if verbose:
            print(" ".join(cmd))
        objs.append(obj)
        procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    logs = [(p.communicate()[0], p.returncode) for p in procs]
    try:
        if any(rc != 0 for _, rc in logs):
            raise DsvcError("nvcc failed:\n" + "".join(l for l, _ in logs))
        r = subprocess.run([nvcc, "-shared", "-o", tmp] + objs, capture_output=True, text=True)
        if r.returncode != 0:
            raise DsvcError("nvcc link failed:\n" + r.stdout + r.stderr)
    finally:
        for o in objs:
            if os.path.exists(o):
                os.remove(o)
    os.replace(tmp, out)
    return out


class DiffnetConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("mel_bins", "residual_channels", "encoder_hidden", "residual_layers",
                                         "dilation_cycle_length", "num_timesteps", "math")]


_FP = C.POINTER(C.c_float)
_FPP = C.POINTER(_FP)


class DiffnetWeights(C.Structure):
    _fields_ = [("input_projection_w", _FP), ("input_projection_b", _FP), ("mlp0_w", _FP), ("mlp0_b", _FP),
                ("mlp2_w", _FP), ("mlp2_b", _FP), ("dilated_conv_w", _FPP), ("dilated_conv_b", _FPP),
                ("diffusion_proj_w", _FPP), ("diffusion_proj_b", _FPP), ("conditioner_proj_w", _FPP),
                ("conditioner_proj_b", _FPP), ("output_proj_w", _FPP), ("output_proj_b", _FPP),
                ("skip_projection_w", _FP), ("skip_projection_b", _FP), ("output_projection_w", _FP),
                ("output_projection_b", _FP), ("step_basis", _FP)]


class NsfConfig(C.Structure):
    _fields_ = [("num_mels", C.c_int32), ("sampling_rate", C.c_int32), ("upsample_initial_channel", C.c_int32),
                ("num_upsamples", C.c_int32), ("upsample_rates", C.c_int32 * MAX_STAGES),
                ("upsample_kernel_sizes", C.c_int32 * MAX_STAGES), ("num_kernels", C.c_int32),
                ("resblock_kernel_sizes", C.c_int32 * MAX_KERNELS), ("num_dilations", C.c_int32),
                ("resblock_dilation_sizes", (C.c_int32 * MAX_DILATIONS) * MAX_KERNELS), ("harmonic_num", C.c_int32),
                ("has_source", C.c_int32)]


class NsfWeights(C.Structure):
    _fields_ = [("source_linear_w", _FP), ("source_linear_b", _FP), ("conv_pre_w", _FP), ("conv_pre_b", _FP),
                ("ups_w", _FPP), ("ups_b", _FPP), ("noise_convs_w", _FPP), ("noise_convs_b", _FPP),
                ("convs1_w", _FPP), ("convs1_b", _FPP), ("convs2_w", _FPP), ("convs2_b", _FPP),
                ("conv_post_w", _FP), ("conv_post_b", _FP)]


class MelConfig(C.Structure):
    _fields_ = [("n_fft", C.c_int32), ("hop_size", C.c_int32), ("n_mels", C.c_int32), ("clip_val", C.c_float),
                ("out_scale", C.c_float)]


class PeConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_mel_bins", "hidden_size", "predictor_hidden", "prenet_layers", "prenet_kernel",
                                         "enc_layers", "enc_kernel", "gn_groups", "pred_layers", "pred_kernel", "pad_same",
                                         "odim", "pos_rows", "pitch_norm", "apply_uv")] + \
               [(n, C.c_float) for n in ("f0_mean", "f0_std", "bn_eps", "gn_eps", "ln_eps")]


class PeWeights(C.Structure):
    _fields_ = [("prenet_conv_w", _FPP), ("prenet_conv_b", _FPP), ("prenet_bn_w", _FPP), ("prenet_bn_b", _FPP),
                ("prenet_bn_mean", _FPP), ("prenet_bn_var", _FPP), ("prenet_out_w", _FP), ("prenet_out_b", _FP),
                ("enc_in_w", _FP), ("enc_in_b", _FP), ("enc_conv_w", _FPP), ("enc_conv_b", _FPP), ("enc_gn_w", _FPP),
                ("enc_gn_b", _FPP), ("enc_out_w", _FP), ("enc_out_b", _FP), ("pred_conv_w", _FPP), ("pred_conv_b", _FPP),
                ("pred_ln_w", _FPP), ("pred_ln_b", _FPP), ("pred_linear_w", _FP), ("pred_linear_b", _FP),
                ("pos_table", _FP), ("pos_embed_alpha", _FP)]


# every symbol include/dsvc.h declares: (name, restype, argtypes)
_VP = C.c_void_p
SYMBOLS = [
    ("dsvc_version", C.c_char_p, []),
    ("dsvc_abi", C.c_uint32, []),
    ("dsvc_last_error", C.c_char_p, []),
    ("dsvc_device_count", C.c_int, []),
    ("dsvc_launch_count", C.c_uint64, []),
    ("dsvc_diffnet_create", C.c_int, [C.POINTER(_VP), C.POINTER(DiffnetConfig), C.POINTER(DiffnetWeights), _VP]),
    ("dsvc_diffnet_destroy", None, [_VP]),
    ("dsvc_diffnet_set_schedule", C.c_int, [_VP] + [_FP] * 6),
    ("dsvc_diffnet_prepare", C.c_int, [_VP, C.c_int32, C.c_int32, C.POINTER(C.c_int32), _VP, _VP]),
    ("dsvc_diffnet_eval", C.c_int, [_VP, _VP, C.c_int32, _VP, _VP]),
    ("dsvc_cond_encode", C.c_int, [_VP, _VP, _VP, _VP, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_float, C.c_float, _VP, _VP, _VP]),
    ("dsvc_diffnet_run_layer", C.c_int, [_VP, C.c_int32, C.c_int32, C.c_int32, _VP]),
    ("dsvc_sample_ddpm", C.c_int, [_VP, _VP, C.c_int32, _VP, C.c_uint64, _VP]),
    ("dsvc_sample_plms", C.c_int, [_VP, _VP, C.c_int32, C.c_int32, _VP]),
    ("dsvc_nsf_create", C.c_int, [C.POINTER(_VP), C.POINTER(NsfConfig), C.POINTER(NsfWeights), _VP]),
    ("dsvc_nsf_create_ex", C.c_int, [C.POINTER(_VP), C.POINTER(NsfConfig), C.c_int32, C.POINTER(NsfWeights), _VP]),
    ("dsvc_nsf_destroy", None, [_VP]),
    ("dsvc_nsf_forward", C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_uint64, C.c_float, _VP, C.c_int32, C.c_int32, _VP]),
    ("dsvc_mel_frames", C.c_int64, [C.POINTER(MelConfig), C.c_int64]),
    ("dsvc_mel_analysis", C.c_int, [C.POINTER(MelConfig), _VP, C.c_int64, _VP, _VP, _VP, _VP, _VP, _VP]),
    ("dsvc_pe_create", C.c_int, [C.POINTER(_VP), C.POINTER(PeConfig), C.POINTER(PeWeights), _VP]),
    ("dsvc_pe_destroy", None, [_VP]),
    ("dsvc_pe_forward", C.c_int, [_VP, _VP, C.c_int32, C.c_int32, _VP, _VP, _VP]),
    ("dsvc_compact_frames", C.c_int, [_VP, _VP, C.c_int32, C.c_int32, C.c_float, C.c_float, _VP, _VP, _VP, _VP]),
]

_lib = None


def load():
    """dlopen libdsvc.so (building it first if the sources are newer) and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("DSVC_LIB")        # developer override (e.g. an instrumented build)
    if not path:
        # Rebuild when the library is missing, or (on the GPU-less build box only) older than its sources.
        # On a GPU box an existing library is used as shipped: N ranks must not race an nvcc rebuild.
        need = not os.path.exists(LIB_PATH)
        if not need and _stale() and os.path.exists("/usr/local/cuda/bin/nvcc"):
            import torch
            need = (not torch.cuda.is_available()) or os.environ.get("DSVC_AUTOBUILD") == "1"
        if need:
            build()
        path = LIB_PATH
    lib = C.CDLL(path)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)           # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    abi = lib.dsvc_abi()
    if abi != 0 and abi != header_crc():
        raise DsvcError("%s was built from another include/dsvc.h (abi %08x, header %08x): rebuild it "
                        "(python -c 'import __graft_entry__ as g; g.build()')" % (path, abi, header_crc()))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise DsvcError("libdsvc error %d: %s" % (rc, load().dsvc_last_error().decode("utf-8", "replace")))


def fptr(t):
    """float* of a contiguous fp32 CPU tensor (the caller keeps `t` alive)."""
    import torch
    assert t.dtype == torch.float32 and t.is_contiguous() and t.device.type == "cpu", (t.dtype, t.device)
    return C.cast(t.data_ptr(), _FP)


def fptr_array(ts):
    arr = (_FP * len(ts))(*[fptr(t) for t in ts])
    return arr


def dptr(t):
    """device pointer of a contiguous CUDA tensor as void*."""
    assert t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA tensor"
    return C.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
