"""ctypes binding of libpkb200.so and the Python mirror of the reference interfaces.

Reference interfaces mirrored here (paths relative to the pocketkaldi tree):
  Fbank            src/fbank.h:46-53     Fbank(), Compute(wave) -> [T][40]
  CMVN             src/cmvn.h:17-26      CMVN(global_stats, raw_feats), GetFrame(t)
  Nnet             src/nnet.h:88-96      Read(file), Propagate(in) -> out
  AcousticModel    src/am.h:21-38        Read(conf), Compute(frames), TransitionIdToPdfId, num_pdfs
  Decodable        src/decodable.h:15-41 init(am, prob_scale, feats), loglikelihood, islastframe
"""

import ctypes as C
import os
import subprocess
import weakref

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpkb200.so")
CSRC = os.path.join(HERE, "csrc")

PREC_BF16, PREC_BF16X3, PREC_FP16 = 0, 1, 2
PREC_FP16X3, PREC_FP16C8, PREC_FP16R = 3, 4, 5
STAGE_FBANK, STAGE_CMVN, STAGE_NNET, STAGE_ALL = 1, 2, 4, 7
STAGE_NO_FEATS = 8  # with STAGE_CMVN + a model: skip the FP32 copy of the CMVN features
BUF_PCM, BUF_RAW, BUF_FEATS, BUF_LOGLIK = 0, 1, 2, 3
BUF_LOGLIK16, BUF_LOGLIK_OFF = 4, 5  # compact output (Batch.set_compact)
KERNEL_CLASSES = ("fbank", "cmvn", "gemm", "gemm_final", "misc")

# pkb_lattice_arc_t (include/pkb200.h)
LATTICE_ARC_DTYPE = np.dtype([("t", np.int32), ("src", np.int32), ("dst", np.int32), ("ilabel", np.int32),
                              ("olabel", np.int32), ("graph_cost", np.float32), ("acoustic_cost", np.float32)])
assert LATTICE_ARC_DTYPE.itemsize == 28
# pkb_frame_post_t (include/pkb200.h)
FRAME_POST_DTYPE = np.dtype([("t", np.int32), ("pdf", np.int32), ("post", np.float32)])
assert FRAME_POST_DTYPE.itemsize == 12

_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_i16p = np.ctypeslib.ndpointer(dtype=np.int16, flags="C_CONTIGUOUS")


class PkbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("pkb error %d: %s" % (code, message))
        self.code = code


def build_library(verbose=False):
    """Compiles libpkb200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j8"]
    if not verbose:
        cmd.insert(1, "-s")
    subprocess.check_call(cmd)
    return LIB_PATH


# Every symbol include/pkb200.h declares: (name, restype, argtypes)
_VP = C.c_void_p
_SIGNATURES = [
    ("pkb_last_error", C.c_char_p, []),
    ("pkb_version", C.c_char_p, []),
    ("pkb_create", C.c_int, [C.c_int, C.POINTER(_VP)]),
    ("pkb_destroy", None, [_VP]),
    ("pkb_sync", C.c_int, [_VP]),
    ("pkb_device_sm_count", C.c_int, [_VP]),
    ("pkb_device_name", C.c_char_p, [_VP]),
    ("pkb_fbank_num_frames", C.c_int, [C.c_int]),
    ("pkb_fbank_set_options", C.c_int, [_VP, C.c_int, C.c_float, C.c_uint64]),
    ("pkb_fbank_f32", C.c_int, [_VP, _f32p, _i32p, C.c_int, _f32p, _i32p]),
    ("pkb_fbank_i16", C.c_int, [_VP, _i16p, _i32p, C.c_int, _f32p, _i32p]),
    ("pkb_cmvn", C.c_int, [_VP, _f32p, _i32p, C.c_int, _f32p, _f32p]),
    ("pkb_am_load", C.c_int, [_VP, C.c_char_p, C.c_int, C.POINTER(_VP)]),
    ("pkb_am_create", C.c_int, [_VP, C.c_int, _i32p, C.POINTER(_VP), C.POINTER(_VP), _i32p, _i32p,
                                _VP, C.c_int, C.c_int, C.c_int, _VP, C.c_int, C.c_int,
                                C.POINTER(_VP)]),
    ("pkb_am_destroy", None, [_VP]),
    ("pkb_am_num_pdfs", C.c_int, [_VP]),
    ("pkb_am_set_refine_margin", C.c_int, [_VP, C.c_float]),
    ("pkb_am_input_dim", C.c_int, [_VP]),
    ("pkb_am_left_context", C.c_int, [_VP]),
    ("pkb_am_right_context", C.c_int, [_VP]),
    ("pkb_am_tid2pdf", C.c_int, [_VP, C.c_int]),
    ("pkb_am_num_tids", C.c_int, [_VP]),
    ("pkb_am_compute", C.c_int, [_VP, _VP, _f32p, _i32p, C.c_int, C.c_int, C.c_float, _f32p]),
    ("pkb_event_create", C.c_int, [_VP, C.POINTER(_VP)]),
    ("pkb_event_destroy", None, [_VP]),
    ("pkb_event_record", C.c_int, [_VP, _VP]),
    ("pkb_event_wait", C.c_int, [_VP]),
    ("pkb_event_query", C.c_int, [_VP, C.POINTER(C.c_int)]),
    ("pkb_am_compute_chunked", C.c_int, [_VP, _VP, _f32p, C.c_int32, C.c_int, C.c_float, _VP, C.c_int,
                                         C.POINTER(_VP), C.c_int]),
    ("pkb_nnet_propagate", C.c_int, [_VP, _VP, _f32p, C.c_int, C.c_int, _f32p]),
    ("pkb_pcm_to_loglik_i16", C.c_int, [_VP, _VP, _i16p, _i32p, C.c_int, _f32p, C.c_float, _VP, _VP,
                                        _VP]),
    ("pkb_batch_create", C.c_int, [_VP, _VP, C.c_int, _i32p, _f32p, C.c_float, C.POINTER(_VP)]),
    ("pkb_batch_destroy", None, [_VP]),
    ("pkb_batch_num_frames", C.c_int64, [_VP]),
    ("pkb_batch_num_samples", C.c_int64, [_VP]),
    ("pkb_batch_set_pcm_i16", C.c_int, [_VP, _VP]),
    ("pkb_batch_synth_pcm", C.c_int, [_VP, C.c_uint64, C.c_uint64]),
    ("pkb_batch_run", C.c_int, [_VP, C.c_int]),
    ("pkb_batch_get", C.c_int, [_VP, C.c_int, _VP]),
    ("pkb_batch_get_rows", C.c_int, [_VP, C.c_int, C.c_int64, C.c_int64, _VP]),
    ("pkb_batch_checksum", C.c_int, [_VP, C.c_int, C.POINTER(C.c_double)]),
    ("pkb_batch_set_compact", C.c_int, [_VP, C.c_int]),
    ("pkb_batch_refine_stats", C.c_int, [_VP, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("pkb_fst_load", C.c_int, [_VP, C.c_char_p, C.POINTER(_VP)]),
    ("pkb_fst_create", C.c_int, [_VP, C.c_int, C.c_int, _VP, _VP, C.c_int, _VP, C.POINTER(_VP)]),
    ("pkb_fst_destroy", None, [_VP]),
    ("pkb_batch_decode", C.c_int, [_VP, _VP, C.c_float, C.c_int, C.c_int, _VP, _VP, _VP]),
    ("pkb_batch_set_max_active", C.c_int, [_VP, C.c_int]),
    ("pkb_batch_lattice", C.c_int, [_VP, _VP, C.c_float, C.c_float, C.c_int, C.c_int, _VP, _VP]),
    ("pkb_batch_lattice_get", C.c_int, [_VP, _VP]),
    ("pkb_batch_nbest", C.c_int, [_VP, _VP, C.c_int, C.c_int, _VP, _VP, _VP, _VP, _VP]),
    ("pkb_batch_posteriors", C.c_int, [_VP, _VP, C.c_float, C.c_float, C.c_float, _VP, _VP]),
    ("pkb_batch_posteriors_get", C.c_int, [_VP, _VP, _VP]),
    ("pkb_batch_best_path", C.c_int, [_VP, _VP, C.c_float, C.c_float, C.c_float, _VP, _VP, _VP, _VP, _VP]),
    ("pkb_batch_best_path_get", C.c_int, [_VP, _VP, _VP, _VP]),
    ("pkb_decoder_create", C.c_int, [_VP, _VP, _VP, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int,
                                     C.POINTER(_VP)]),
    ("pkb_decoder_destroy", None, [_VP]),
    ("pkb_decoder_advance", C.c_int, [_VP, _VP, C.c_int, _VP]),
    ("pkb_decoder_partial", C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    ("pkb_decoder_finish", C.c_int, [_VP, _VP, _VP, _VP]),
    ("pkb_decoder_set_lattice", C.c_int, [_VP, C.c_float, C.c_int, C.c_int]),
    ("pkb_decoder_set_max_active", C.c_int, [_VP, C.c_int]),
    ("pkb_decoder_lattice", C.c_int, [_VP, _VP, _VP]),
    ("pkb_decoder_lattice_get", C.c_int, [_VP, _VP]),
    ("pkb_decoder_nbest", C.c_int, [_VP, C.c_int, C.c_int, _VP, _VP, _VP, _VP, _VP]),
    ("pkb_decoder_posteriors", C.c_int, [_VP, C.c_float, C.c_float, C.c_float, _VP, _VP]),
    ("pkb_decoder_posteriors_get", C.c_int, [_VP, _VP, _VP]),
    ("pkb_decoder_best_path", C.c_int, [_VP, C.c_float, C.c_float, C.c_float, _VP, _VP, _VP, _VP, _VP]),
    ("pkb_decoder_best_path_get", C.c_int, [_VP, _VP, _VP, _VP]),
    ("pkb_loglik16_expand", C.c_int, [_VP, _VP, C.c_int64, C.c_int, C.c_float, _VP]),
    ("pkb_stream_create", C.c_int, [_VP, _VP, C.c_int, C.c_int, _f32p, C.c_float, C.POINTER(_VP)]),
    ("pkb_stream_destroy", None, [_VP]),
    ("pkb_stream_max_frames", C.c_int, [_VP]),
    ("pkb_stream_push_i16", C.c_int, [_VP, _VP, _VP, _VP]),
    ("pkb_stream_flush", C.c_int, [_VP, _VP, _VP]),
    ("pkb_stream_set_compact", C.c_int, [_VP, C.c_int]),
    ("pkb_stream_graph_replays", C.c_int, [_VP, C.POINTER(C.c_int64)]),
    ("pkb_stream_push_compact_i16", C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    ("pkb_stream_flush_compact", C.c_int, [_VP, _VP, _VP, _VP]),
    ("pkb_stream_set_decoder", C.c_int, [_VP, _VP]),
    ("pkb_wav_probe", C.c_int, [C.c_char_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("pkb_wav_read_i16", C.c_int, [C.c_char_p, _VP, C.c_int32, C.POINTER(C.c_int32)]),
    ("pkb_wav_read_f32", C.c_int, [C.c_char_p, _VP, C.c_int32, C.POINTER(C.c_int32)]),
    ("pkb_scp_open", C.c_int, [C.c_char_p, C.POINTER(_VP)]),
    ("pkb_wavlist_create", C.c_int, [C.POINTER(C.c_char_p), C.c_int, C.POINTER(_VP)]),
    ("pkb_wavlist_destroy", None, [_VP]),
    ("pkb_wavlist_size", C.c_int, [_VP]),
    ("pkb_wavlist_path", C.c_char_p, [_VP, C.c_int]),
    ("pkb_wavlist_num_samples", C.POINTER(C.c_int32), [_VP]),
    ("pkb_wavlist_read_i16", C.c_int, [_VP, C.c_int, C.c_int, _VP, C.c_int]),
    ("pkb_host_alloc", C.c_int, [C.POINTER(_VP), C.c_uint64]),
    ("pkb_host_free", None, [_VP]),
    ("pkb_timer_start", C.c_int, [_VP]),
    ("pkb_timer_stop", C.c_int, [_VP, C.POINTER(C.c_float)]),
    ("pkb_profile_enable", C.c_int, [_VP, C.c_int]),
    ("pkb_profile_reset", C.c_int, [_VP]),
    ("pkb_profile_get", C.c_int, [_VP, C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    ("pkb_flush_l2", C.c_int, [_VP]),
]
EXPORTED_SYMBOLS = [s[0] for s in _SIGNATURES]

_lib = None


def load_library():
    """Loads libpkb200.so (no GPU needed to load). Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PkbError(-1, "%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, restype, argtypes in _SIGNATURES:
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def _check(rc):
    if rc != 0:
        raise PkbError(rc, load_library().pkb_last_error().decode("utf-8", "replace"))


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _lens(lens):
    return np.ascontiguousarray(lens, dtype=np.int32)


class PinnedArray:
    """numpy view over page-locked host memory from pkb_host_alloc."""

    def __init__(self, shape, dtype):
        self.lib = load_library()
        self.ptr = _VP()
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        _check(self.lib.pkb_host_alloc(C.byref(self.ptr), max(n, 1)))
        buf = (C.c_char * max(n, 1)).from_address(self.ptr.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self.ptr:
            self.array = None
            self.lib.pkb_host_free(self.ptr)
            self.ptr = None


def read_wav(path, dtype=np.float32):
    """pk_16kpcm_read (src/pcm_reader.cc:45-220): strict 16 kHz mono PCM WAV -> unscaled samples.
    dtype float32 gives exactly the reference's vector; int16 is the batch pipeline's input."""
    lib = load_library()
    n = C.c_int32(0)
    bits = C.c_int32(0)
    _check(lib.pkb_wav_probe(os.fsencode(path), C.byref(n), C.byref(bits)))
    out = np.empty(n.value, dtype=dtype)
    fn = {np.dtype(np.float32): lib.pkb_wav_read_f32, np.dtype(np.int16): lib.pkb_wav_read_i16}[np.dtype(dtype)]
    _check(fn(os.fsencode(path), out.ctypes.data_as(_VP), n.value, C.byref(n)))
    return out


class WavList:
    """A validated list of wave files (pkb_wavlist_t): `.scp` file or a sequence of paths.
    Replaces the one-file-at-a-time loop of src/main.cc:34-46 for the batch pipeline."""

    def __init__(self, scp_or_paths):
        self.lib = load_library()
        self.h = _VP()
        if isinstance(scp_or_paths, (str, bytes, os.PathLike)):
            _check(self.lib.pkb_scp_open(os.fsencode(scp_or_paths), C.byref(self.h)))
        else:
            enc = [os.fsencode(p) for p in scp_or_paths]
            arr = (C.c_char_p * max(len(enc), 1))(*enc)
            _check(self.lib.pkb_wavlist_create(arr, len(enc), C.byref(self.h)))

    def close(self):
        if self.h:
            self.lib.pkb_wavlist_destroy(self.h)
            self.h = None

    def __len__(self):
        return self.lib.pkb_wavlist_size(self.h)

    def path(self, i):
        p = self.lib.pkb_wavlist_path(self.h, i)
        if p is None:
            raise IndexError(i)
        return os.fsdecode(p)

    @property
    def num_samples(self):
        n = len(self)
        if n == 0:
            return np.zeros(0, np.int32)
        return np.ctypeslib.as_array(self.lib.pkb_wavlist_num_samples(self.h), shape=(n,)).copy()

    def read_i16(self, first=0, count=None, out=None, n_threads=0):
        """Samples of files [first, first+count) back to back (the pkb_batch_set_pcm_i16 layout).
        `out` may be a PinnedArray's .array."""
        count = len(self) - first if count is None else count
        total = int(self.num_samples[first:first + count].sum())
        if out is None:
            out = np.empty(total, np.int16)
        assert out.dtype == np.int16 and out.size >= total and out.flags["C_CONTIGUOUS"]
        _check(self.lib.pkb_wavlist_read_i16(self.h, first, count, out.ctypes.data_as(_VP), n_threads))
        return out[:total]


class Context:
    """One per GPU (pkb_ctx_t): stream, front-end tables, scratch."""

    def __init__(self, device=0):
        self.lib = load_library()
        self.h = _VP()
        self._children = weakref.WeakSet()
        _check(self.lib.pkb_create(device, C.byref(self.h)))

    def _adopt(self, child):
        """Objects created on this context are closed before it (the C ABI requires that order)."""
        self._children.add(child)

    def close(self):
        if self.h:
            kids = list(self._children)
            for child in sorted(kids, key=lambda k: isinstance(k, AcousticModel)):  # models last
                child.close()
            self.lib.pkb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self):
        _check(self.lib.pkb_sync(self.h))

    @property
    def sm_count(self):
        return self.lib.pkb_device_sm_count(self.h)

    @property
    def device_name(self):
        return self.lib.pkb_device_name(self.h).decode()

    def timer_start(self):
        _check(self.lib.pkb_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float(0)
        _check(self.lib.pkb_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def profile_enable(self, on):
        _check(self.lib.pkb_profile_enable(self.h, 1 if on else 0))

    def profile_reset(self):
        _check(self.lib.pkb_profile_reset(self.h))

    def profile_get(self):
        n = len(KERNEL_CLASSES)
        launches = (C.c_int64 * n)()
        ms = (C.c_double * n)()
        _check(self.lib.pkb_profile_get(self.h, launches, ms))
        return {k: (int(launches[i]), float(ms[i])) for i, k in enumerate(KERNEL_CLASSES)}

    def set_fbank_options(self, window="hamming", dither=0.0, dither_seed=0):
        """Front-end options the reference does not have (pkb_fbank_set_options): parity unpinned."""
        _check(self.lib.pkb_fbank_set_options(self.h, {"hamming": 0, "povey": 1}[window], dither,
                                              dither_seed))

    def flush_l2(self):
        _check(self.lib.pkb_flush_l2(self.h))

    # ---- batched front end
    def fbank_batch(self, waves):
        """waves: list of 1-D arrays (float32 int16-range samples, or int16). -> list of [T][40]."""
        lens = _lens([len(w) for w in waves])
        is_i16 = all(np.asarray(w).dtype == np.int16 for w in waves) and len(waves) > 0
        dt = np.int16 if is_i16 else np.float32
        flat = (np.concatenate([np.asarray(w, dtype=dt) for w in waves]) if len(waves)
                else np.zeros(0, dt))
        flat = np.ascontiguousarray(flat if flat.size else np.zeros(1, dt))
        T = np.zeros(max(len(waves), 1), np.int32)
        total = int(sum(self.lib.pkb_fbank_num_frames(int(n)) for n in lens))
        out = np.empty((max(total, 1), 40), np.float32)
        fn = self.lib.pkb_fbank_i16 if is_i16 else self.lib.pkb_fbank_f32
        _check(fn(self.h, flat, lens if len(waves) else np.zeros(1, np.int32), len(waves), out, T))
        res, o = [], 0
        for u in range(len(waves)):
            res.append(out[o:o + T[u]].copy())
            o += int(T[u])
        return res

    def cmvn_batch(self, raws, global_stats):
        lens = _lens([r.shape[0] for r in raws])
        total = int(lens.sum()) if len(raws) else 0
        flat = _f32(np.concatenate([_f32(r).reshape(-1, 40) for r in raws]) if total
                    else np.zeros((1, 40), np.float32))
        out = np.empty_like(flat)
        _check(self.lib.pkb_cmvn(self.h, flat, lens if len(raws) else np.zeros(1, np.int32),
                                 len(raws), _f32(global_stats), out))
        res, o = [], 0
        for n in lens:
            res.append(out[o:o + n].copy())
            o += int(n)
        return res


class Fbank:
    """pocketkaldi::Fbank (src/fbank.h:46-53)."""

    def __init__(self, ctx):
        self.ctx = ctx

    def CalcNumFrames(self, num_samples):
        return self.ctx.lib.pkb_fbank_num_frames(int(num_samples))

    def Compute(self, wave):
        """wave: float32 samples in int16 range (pk_16kpcm_read output) or int16. -> [T][40]."""
        return self.ctx.fbank_batch([np.asarray(wave)])[0]


class CMVN:
    """pocketkaldi::CMVN (src/cmvn.h:17-26). The whole utterance is normalised on the GPU at
    construction; GetFrame(t) must be called in order as in the reference (src/cmvn.cc:38)."""

    def __init__(self, ctx, global_stats, raw_feats):
        self.feats = ctx.cmvn_batch([_f32(raw_feats)], global_stats)[0]
        self._cached_frame = -1

    def GetFrame(self, frame):
        assert self._cached_frame == frame - 1, "frames must be requested in order"
        self._cached_frame = frame
        return self.feats[frame]


class AcousticModel:
    """pocketkaldi::AcousticModel (src/am.h:21-38) resident on the GPU."""

    def __init__(self, ctx, precision=PREC_BF16X3):
        self.ctx = ctx
        self.precision = precision
        self.h = None
        ctx._adopt(self)

    def Read(self, conf_path):
        """AcousticModel::Read(conf) (src/am.cc:23-63)."""
        h = _VP()
        _check(self.ctx.lib.pkb_am_load(self.ctx.h, conf_path.encode(), self.precision, C.byref(h)))
        self._replace(h)
        return self

    def from_layers(self, layers, prior, left, right, tid2pdf=None):
        """layers: as pocketkaldi_b200.formats.read_nnet returns them (MUL layers are folded
        the way the file loader folds them)."""
        if any(l[0] == "mul" for l in layers):
            from .formats import fold_mul_layers
            layers = fold_mul_layers(layers)
        names = {"linear": 0, "relu": 1, "normalize": 2, "softmax": 3, "sigmoid": 6}
        types = np.array([names[l[0]] for l in layers], np.int32)
        Ws = [_f32(l[1]) for l in layers if l[0] == "linear"]
        bs = [_f32(l[2]) for l in layers if l[0] == "linear"]
        n = len(Ws)
        Wp = (_VP * max(n, 1))(*[w.ctypes.data for w in Ws])
        bp = (_VP * max(n, 1))(*[b.ctypes.data for b in bs])
        od = np.array([w.shape[0] for w in Ws], np.int32)
        idm = np.array([w.shape[1] for w in Ws], np.int32)
        pr = _f32(prior) if prior is not None else None
        t2p = np.ascontiguousarray(tid2pdf, dtype=np.int32) if tid2pdf is not None else None
        h = _VP()
        _check(self.ctx.lib.pkb_am_create(
            self.ctx.h, len(types), types, Wp, bp, od, idm,
            pr.ctypes.data if pr is not None else None, len(pr) if pr is not None else 0,
            left, right, t2p.ctypes.data if t2p is not None else None,
            len(t2p) if t2p is not None else 0, self.precision, C.byref(h)))
        self._replace(h)
        self._keep = (Ws, bs, pr, t2p)
        return self

    def _replace(self, h):
        self.close()
        self.h = h

    def close(self):
        if self.h:
            self.ctx.lib.pkb_am_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def num_pdfs(self):
        return self.ctx.lib.pkb_am_num_pdfs(self.h)

    def set_refine_margin(self, margin):
        """PREC_FP16R: frames whose two best pdfs are closer than `margin` are recomputed."""
        _check(self.ctx.lib.pkb_am_set_refine_margin(self.h, float(margin)))

    def input_dim(self):
        return self.ctx.lib.pkb_am_input_dim(self.h)

    def TransitionIdToPdfId(self, tid):
        return self.ctx.lib.pkb_am_tid2pdf(self.h, int(tid))

    def Compute(self, frames, prob_scale=1.0):
        """AcousticModel::Compute (src/am.cc:90-115). frames: [T][feat_dim] -> [T][num_pdfs]."""
        return self.compute_batch([frames], prob_scale)[0]

    def compute_batch(self, feats_list, prob_scale=1.0):
        lens = _lens([f.shape[0] for f in feats_list])
        total = int(lens.sum()) if len(feats_list) else 0
        dim = feats_list[0].shape[1] if len(feats_list) else 0
        P = self.num_pdfs()
        flat = _f32(np.concatenate([_f32(f) for f in feats_list]) if total
                    else np.zeros((1, max(dim, 1)), np.float32))
        out = np.empty((max(total, 1), P), np.float32)
        _check(self.ctx.lib.pkb_am_compute(self.ctx.h, self.h, flat,
                                           lens if len(feats_list) else np.zeros(1, np.int32),
                                           len(feats_list), dim, prob_scale, out))
        res, o = [], 0
        for n in lens:
            res.append(out[o:o + n].copy())
            o += int(n)
        return res

    def pcm_to_loglik(self, pcms, global_stats, prob_scale=1.0, want_feats=False):
        """Fused pk_process front half (src/pocketkaldi.cc:192-216) on int16 PCM."""
        lens = _lens([len(p) for p in pcms])
        flat = np.ascontiguousarray(np.concatenate([np.asarray(p, np.int16) for p in pcms]))
        T = np.zeros(len(pcms), np.int32)
        total = int(sum(self.ctx.lib.pkb_fbank_num_frames(int(n)) for n in lens))
        P = self.num_pdfs()
        ll = np.empty((max(total, 1), P), np.float32)
        ft = np.empty((max(total, 1), 40), np.float32) if want_feats else None
        _check(self.ctx.lib.pkb_pcm_to_loglik_i16(
            self.ctx.h, self.h, flat, lens, len(pcms), _f32(global_stats), prob_scale,
            ll.ctypes.data, ft.ctypes.data if ft is not None else None, T.ctypes.data))
        res, fres, o = [], [], 0
        for n in T:
            res.append(ll[o:o + n].copy())
            if ft is not None:
                fres.append(ft[o:o + n].copy())
            o += int(n)
        return (res, fres) if want_feats else res


class Nnet:
    """pocketkaldi::Nnet (src/nnet.h:88-96): the layer stack without splice or prior."""

    def __init__(self, ctx, precision=PREC_BF16X3):
        self.ctx = ctx
        self.am = AcousticModel(ctx, precision)

    def Read(self, nnet_path):
        from . import formats
        return self.from_layers(formats.read_nnet(nnet_path))

    def from_layers(self, layers):
        self.am.from_layers(layers, None, 0, 0)
        return self

    def Propagate(self, x):
        x = _f32(x)
        rows, dim = x.shape
        lin = self.am
        out_dim = lin.num_pdfs()
        out = np.empty((max(rows, 1), out_dim), np.float32)
        _check(self.ctx.lib.pkb_nnet_propagate(self.ctx.h, lin.h, x if rows else np.zeros((1, dim), np.float32),
                                               rows, dim, out))
        return out[:rows]


class Event:
    """pkb_event_t: a point of the context's stream the host can wait for."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.h = _VP()
        _check(ctx.lib.pkb_event_create(ctx.h, C.byref(self.h)))
        ctx._adopt(self)

    def record(self):
        _check(self.ctx.lib.pkb_event_record(self.ctx.h, self.h))

    def wait(self):
        _check(self.ctx.lib.pkb_event_wait(self.h))

    def done(self):
        d = C.c_int(0)
        _check(self.ctx.lib.pkb_event_query(self.h, C.byref(d)))
        return bool(d.value)

    def close(self):
        if self.h:
            self.ctx.lib.pkb_event_destroy(self.h)
            self.h = None


class Decodable:
    """pk_decodable_t (src/decodable.h:15-41): AM evaluation + table look-up.

    chunk_frames = 0: eager like the reference (pk_decodable_init returns when the whole matrix
    is on the host). chunk_frames > 0: lazy (SURVEY 8(f)-1) -- the matrix lands in page-locked
    memory chunk by chunk and loglikelihood(frame, ...) only waits for the chunk holding `frame`,
    so a frame-synchronous decoder (src/decoder.cc:49) starts after the first chunk."""

    def __init__(self, am, prob_scale, feats, chunk_frames=0):
        self.am = am
        self._events = []
        self._pinned = None
        if chunk_frames <= 0:
            self.log_prob = am.Compute(feats, prob_scale)  # pk_decodable_init
            self._ready = self.log_prob.shape[0]
            return
        feats = _f32(feats)
        T, P = feats.shape[0], am.num_pdfs()
        self._chunk = chunk_frames
        self._pinned = PinnedArray((max(T, 1), P), np.float32)
        self.log_prob = self._pinned.array[:T]
        self._events = [Event(am.ctx) for _ in range((T + chunk_frames - 1) // chunk_frames)]
        self._ready = 0
        arr = (_VP * max(len(self._events), 1))(*[e.h for e in self._events])
        _check(am.ctx.lib.pkb_am_compute_chunked(am.ctx.h, am.h, feats if T else np.zeros((1, 1), np.float32),
                                                 T, feats.shape[1], prob_scale,
                                                 self._pinned.array.ctypes.data_as(_VP), chunk_frames,
                                                 arr, len(self._events)))

    def frames_ready(self):
        """Frames whose log-likelihoods are already in host memory (non-blocking)."""
        while self._ready < self.log_prob.shape[0] and self._events[self._ready // self._chunk].done():
            self._ready = min(self.log_prob.shape[0], (self._ready // self._chunk + 1) * self._chunk)
        return self._ready

    def loglikelihood(self, frame, trans_id):
        if frame >= self._ready:
            self._events[frame // self._chunk].wait()   # stream order: earlier chunks are done too
            self._ready = min(self.log_prob.shape[0], (frame // self._chunk + 1) * self._chunk)
        return float(self.log_prob[frame, self.am.TransitionIdToPdfId(trans_id)])

    def islastframe(self, frame):
        assert frame < self.log_prob.shape[0]
        return frame == self.log_prob.shape[0] - 1

    def close(self):
        if self._events:
            self._events[-1].wait()
        for e in self._events:
            e.close()
        self._events = []
        if self._pinned is not None:
            self.log_prob = None
            self._pinned.free()
            self._pinned = None


class Batch:
    """Device-resident utterance batch (pkb_batch_t): the throughput pipeline."""

    def __init__(self, ctx, num_samples, global_stats, am=None, prob_scale=1.0):
        self.ctx = ctx
        self.am = am
        self.num_samples = _lens(num_samples)
        self.h = _VP()
        _check(ctx.lib.pkb_batch_create(ctx.h, am.h if am is not None else None,
                                        len(self.num_samples), self.num_samples,
                                        _f32(global_stats), prob_scale, C.byref(self.h)))
        self.num_frames = np.array([ctx.lib.pkb_fbank_num_frames(int(n)) for n in self.num_samples],
                                   np.int64)
        ctx._adopt(self)

    def close(self):
        if self.h:
            self.ctx.lib.pkb_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def total_frames(self):
        return int(self.ctx.lib.pkb_batch_num_frames(self.h))

    @property
    def total_samples(self):
        return int(self.ctx.lib.pkb_batch_num_samples(self.h))

    def set_pcm(self, pcm_flat):
        """pcm_flat: contiguous int16 array (numpy or PinnedArray.array) of all samples."""
        assert pcm_flat.dtype == np.int16 and pcm_flat.size == self.total_samples
        _check(self.ctx.lib.pkb_batch_set_pcm_i16(self.h, pcm_flat.ctypes.data))

    def synth_pcm(self, seed, first_utt_id=0):
        _check(self.ctx.lib.pkb_batch_synth_pcm(self.h, seed, first_utt_id))

    def run(self, stages=STAGE_ALL):
        _check(self.ctx.lib.pkb_batch_run(self.h, stages))

    def _shape(self, which):
        if which == BUF_PCM:
            return (self.total_samples,), np.int16
        if which in (BUF_RAW, BUF_FEATS):
            return (self.total_frames, 40), np.float32
        if which == BUF_LOGLIK16:
            return (self.total_frames, self.am.num_pdfs()), np.uint16
        if which == BUF_LOGLIK_OFF:
            return (self.total_frames,), np.float32
        return (self.total_frames, self.am.num_pdfs()), np.float32

    def decode(self, fst, beam=0.0, max_tokens=0, max_words=256):
        """GPU Viterbi over the batch's FP32 log-likelihoods (pkb_batch_decode): returns
        ([word id lists in spoken order], weights); a failed search gives None for its utterance."""
        n = len(self.num_samples)
        words = np.zeros((max(n, 1), max_words), np.int32)
        nw = np.zeros(max(n, 1), np.int32)
        wt = np.zeros(max(n, 1), np.float32)
        _check(self.ctx.lib.pkb_batch_decode(self.h, fst.h, beam, max_tokens, max_words, words.ctypes.data,
                                             nw.ctypes.data, wt.ctypes.data))
        hyps = [None if nw[u] < 0 else [int(x) for x in words[u, :min(int(nw[u]), max_words)]] for u in range(n)]
        return hyps, wt[:n].copy()

    def set_max_active(self, max_active):
        """Expand at most max_active tokens per frame (ties at the cutoff included) in the later
        decode() and lattice() calls (pkb_batch_set_max_active); 0 switches the limit off."""
        _check(self.ctx.lib.pkb_batch_set_max_active(self.h, max_active))

    def lattice(self, fst, lattice_beam=8.0, beam=0.0, max_tokens=0, max_arcs=0):
        """The search of decode() keeping its lattice pruned to lattice_beam (pkb_batch_lattice):
        returns ([LATTICE_ARC_DTYPE array per utterance, None where the search failed],
        best costs as float64)."""
        lib = self.ctx.lib
        lats, best, self._lat_n = _lattices(
            len(self.num_samples),
            lambda na, bc: lib.pkb_batch_lattice(self.h, fst.h, beam, lattice_beam, max_tokens, max_arcs, na, bc),
            lambda arcs: lib.pkb_batch_lattice_get(self.h, arcs))
        return lats, best

    def nbest(self, fst, n=10, max_words=256):
        """N-best lists of distinct word sequences over the latest lattice() (pkb_batch_nbest; fst
        is the graph of that call): per utterance None where its lattice failed, otherwise a list
        of (words, graph_cost, acoustic_cost), best first."""
        return _nbest(len(self.num_samples), n, max_words,
                      lambda *out: self.ctx.lib.pkb_batch_nbest(self.h, fst.h, n, max_words, *out))

    def posteriors(self, fst, acoustic_scale=1.0, graph_scale=1.0, min_post=0.0):
        """Arc and frame posteriors over the latest lattice() (pkb_batch_posteriors; fst is the graph
        of that call): (totals as float64, per utterance the float32 posteriors of its lattice()
        records or None where its lattice failed, per utterance a FRAME_POST_DTYPE array of its
        (t, pdf) entries or None where its lattice or its posteriors failed)."""
        lib = self.ctx.lib
        return _posteriors(getattr(self, "_lat_n", np.zeros(0, np.int64)), len(self.num_samples),
                           lambda tot, npost: lib.pkb_batch_posteriors(self.h, fst.h, acoustic_scale, graph_scale,
                                                                      min_post, tot, npost),
                           lambda arc, fr: lib.pkb_batch_posteriors_get(self.h, arc, fr))

    def best_path(self, fst, acoustic_scale=1.0, graph_scale=1.0, word_penalty=0.0):
        """The best path of every utterance's latest lattice() at these scales and word insertion
        penalty (pkb_batch_best_path; fst is the graph of that call): per utterance None where its
        lattice or its best path failed, otherwise (cost, graph_cost, acoustic_cost, words as int32,
        word_t as int32, alignment as int32 transition ids, one per frame)."""
        lib = self.ctx.lib
        return _best_path(len(self.num_samples),
                          lambda *out: lib.pkb_batch_best_path(self.h, fst.h, acoustic_scale, graph_scale,
                                                               word_penalty, *out),
                          lambda *out: lib.pkb_batch_best_path_get(self.h, *out))

    def refine_stats(self):
        """(GEMM rows, frames recomputed) of the latest run under PREC_FP16R."""
        rows, sel = C.c_int64(0), C.c_int64(0)
        _check(self.ctx.lib.pkb_batch_refine_stats(self.h, C.byref(rows), C.byref(sel)))
        return rows.value, sel.value

    def set_compact(self, on=True):
        """Half-size output of the nnet stage (see pkb_batch_set_compact in include/pkb200.h)."""
        _check(self.ctx.lib.pkb_batch_set_compact(self.h, 1 if on else 0))

    def expand_compact(self, h16, off, prob_scale):
        """prob_scale * (half(h16) + off[:, None]) through the library's host helper."""
        h16 = np.ascontiguousarray(h16, dtype=np.uint16)
        off = np.ascontiguousarray(off, dtype=np.float32)
        out = np.empty(h16.shape, np.float32)
        _check(self.ctx.lib.pkb_loglik16_expand(h16.ctypes.data, off.ctypes.data, h16.shape[0],
                                                h16.shape[1], prob_scale, out.ctypes.data))
        return out

    def get(self, which, out=None):
        shape, dt = self._shape(which)
        if out is None:
            out = np.empty(shape, dt)
        _check(self.ctx.lib.pkb_batch_get(self.h, which, out.ctypes.data))
        self.ctx.sync()
        return out

    def get_rows_async(self, which, row0, n_rows, out):
        _check(self.ctx.lib.pkb_batch_get_rows(self.h, which, row0, n_rows, out.ctypes.data))

    def checksum(self, which):
        s = C.c_double(0)
        _check(self.ctx.lib.pkb_batch_checksum(self.h, which, C.byref(s)))
        return s.value


class Fst:
    """pocketkaldi::Fst (src/fst.cc:29-129) resident on the GPU for Batch.decode."""

    def __init__(self, ctx, path=None, graph=None):
        """path: a "pk::fst_0" file, or graph = (num_states, start, {state: final weight},
        [(src, dst, ilabel, olabel, weight)]) as pocketkaldi_b200.formats.write_fst takes it."""
        self.ctx = ctx
        self.h = _VP()
        if path is not None:
            _check(ctx.lib.pkb_fst_load(ctx.h, path.encode(), C.byref(self.h)))
        else:
            ns, start, finals, arcs = graph
            arcs = sorted(arcs)
            first = np.full(ns, -1, np.int32)
            for i, a in enumerate(arcs):
                if first[a[0]] == -1:
                    first[a[0]] = i
            fin = np.full(ns, np.inf, np.float32)
            for st, wgt in finals.items():
                fin[st] = wgt
            raw = np.zeros((max(len(arcs), 1), 4), np.int32)
            for i, a in enumerate(arcs):
                raw[i, :3] = (a[1], a[2], a[3])
                raw[i, 3] = np.float32(a[4]).view(np.int32)
            _check(ctx.lib.pkb_fst_create(ctx.h, ns, start, fin.ctypes.data, first.ctypes.data, len(arcs),
                                          raw.ctypes.data, C.byref(self.h)))
        ctx._adopt(self)

    def close(self):
        if self.h:
            self.ctx.lib.pkb_fst_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _hyps(words, nw, max_words):
    return [None if n < 0 else [int(x) for x in words[s, :min(int(n), max_words)]] for s, n in enumerate(nw)]


class Decoder:
    """pkb_decoder_t: n_streams GPU Viterbi searches that advance chunk by chunk. Rows may arrive in
    any split; the result equals Batch.decode over the same rows, bit for bit."""

    def __init__(self, ctx, am, fst, n_streams, beam=0.0, max_tokens=0, max_words=256, max_records=0):
        self.ctx, self.n_streams, self.max_words = ctx, n_streams, max_words
        self.P = am.num_pdfs()
        self.h = _VP()
        _check(ctx.lib.pkb_decoder_create(ctx.h, am.h, fst.h, n_streams, beam, max_tokens, max_words,
                                          max_records, C.byref(self.h)))
        ctx._adopt(self)

    def close(self):
        if self.h:
            self.ctx.lib.pkb_decoder_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def advance(self, loglik, n_frames=None):
        """loglik: float32 [n_streams][frame_stride][num_pdfs]; stream s decodes its first
        n_frames[s] rows (all of them when n_frames is None)."""
        loglik = _f32(loglik)
        assert loglik.ndim == 3 and loglik.shape[0] == self.n_streams and loglik.shape[2] == self.P
        nf = _lens(np.full(self.n_streams, loglik.shape[1]) if n_frames is None else n_frames)
        _check(self.ctx.lib.pkb_decoder_advance(self.h, loglik.ctypes.data if loglik.size else None,
                                                loglik.shape[1], nf.ctypes.data))

    def partial(self):
        """Best-so-far per stream: (word lists or None where the search failed, costs, frames)."""
        words = np.zeros((self.n_streams, self.max_words), np.int32)
        nw = np.zeros(self.n_streams, np.int32)
        cost = np.zeros(self.n_streams, np.float32)
        frames = np.zeros(self.n_streams, np.int64)
        _check(self.ctx.lib.pkb_decoder_partial(self.h, words.ctypes.data, nw.ctypes.data, cost.ctypes.data,
                                                frames.ctypes.data))
        return _hyps(words, nw, self.max_words), cost, frames

    def finish(self):
        """BestPath per stream (as Batch.decode: word lists, None where the search failed, and
        weights), then fresh utterances."""
        words = np.zeros((self.n_streams, self.max_words), np.int32)
        nw = np.zeros(self.n_streams, np.int32)
        wt = np.zeros(self.n_streams, np.float32)
        _check(self.ctx.lib.pkb_decoder_finish(self.h, words.ctypes.data, nw.ctypes.data, wt.ctypes.data))
        return _hyps(words, nw, self.max_words), wt

    def set_lattice(self, lattice_beam=8.0, max_frames=0, max_arcs=0):
        """Every finish() also keeps each stream's lattice pruned to lattice_beam, equal to
        Batch.lattice over the same rows (pkb_decoder_set_lattice); 0 switches lattices off. Only
        between utterances."""
        _check(self.ctx.lib.pkb_decoder_set_lattice(self.h, lattice_beam, max_frames, max_arcs))

    def set_max_active(self, max_active):
        """Batch.set_max_active for the decoder's streams (pkb_decoder_set_max_active). Only between
        utterances."""
        _check(self.ctx.lib.pkb_decoder_set_max_active(self.h, max_active))

    def lattice(self):
        """The lattices of the latest finish(): ([LATTICE_ARC_DTYPE array per stream, None where it
        failed], best costs as float64), as Batch.lattice returns them."""
        lib = self.ctx.lib
        lats, best, _ = _lattices(self.n_streams, lambda na, bc: lib.pkb_decoder_lattice(self.h, na, bc),
                                  lambda arcs: lib.pkb_decoder_lattice_get(self.h, arcs))
        return lats, best

    def nbest(self, n=10, max_words=256):
        """Batch.nbest over the lattices of the latest finish() (pkb_decoder_nbest)."""
        return _nbest(self.n_streams, n, max_words,
                      lambda *out: self.ctx.lib.pkb_decoder_nbest(self.h, n, max_words, *out))

    def posteriors(self, acoustic_scale=1.0, graph_scale=1.0, min_post=0.0):
        """Batch.posteriors over the lattices of the latest finish() (pkb_decoder_posteriors)."""
        lib = self.ctx.lib
        na = np.zeros(self.n_streams, np.int64)
        best = np.zeros(self.n_streams, np.float64)
        _check(lib.pkb_decoder_lattice(self.h, na.ctypes.data, best.ctypes.data))
        return _posteriors(na, self.n_streams,
                           lambda tot, npost: lib.pkb_decoder_posteriors(self.h, acoustic_scale, graph_scale,
                                                                        min_post, tot, npost),
                           lambda arc, fr: lib.pkb_decoder_posteriors_get(self.h, arc, fr))

    def best_path(self, acoustic_scale=1.0, graph_scale=1.0, word_penalty=0.0):
        """Batch.best_path over the lattices of the latest finish() (pkb_decoder_best_path)."""
        lib = self.ctx.lib
        return _best_path(self.n_streams,
                          lambda *out: lib.pkb_decoder_best_path(self.h, acoustic_scale, graph_scale, word_penalty,
                                                                 *out),
                          lambda *out: lib.pkb_decoder_best_path_get(self.h, *out))


def _split(flat, counts):
    """Per utterance the next max(counts[u], 0) entries of flat, or None where counts[u] < 0."""
    off = np.concatenate([[0], np.cumsum(np.maximum(counts, 0))])
    return [None if counts[u] < 0 else flat[off[u]:off[u + 1]].copy() for u in range(len(counts))]


def _lattices(n_utts, call, get):
    """Runs call(n_arcs, best_costs) and get(records) for n_utts utterances and unpacks them as
    Batch.lattice returns them, with the record counts."""
    na = np.zeros(max(n_utts, 1), np.int64)
    best = np.zeros(max(n_utts, 1), np.float64)
    _check(call(na.ctypes.data, best.ctypes.data))
    na = na[:n_utts].copy()
    arcs = np.empty(max(int(np.maximum(na, 0).sum()), 1), LATTICE_ARC_DTYPE)
    _check(get(arcs.ctypes.data))
    return _split(arcs, na), best[:n_utts].copy(), na


def _nbest(n_utts, n, max_words, call):
    """Runs call(words, n_words, graph, acoustic, n_hyps) over output arrays for n_utts utterances and
    unpacks them as Batch.nbest returns them."""
    u = max(n_utts, 1)
    words = np.zeros((u, max(n, 1), max(max_words, 1)), np.int32)
    nw = np.zeros((u, max(n, 1)), np.int32)
    g = np.zeros((u, max(n, 1)), np.float64)
    a = np.zeros((u, max(n, 1)), np.float64)
    nh = np.zeros(u, np.int32)
    _check(call(words.ctypes.data, nw.ctypes.data, g.ctypes.data, a.ctypes.data, nh.ctypes.data))
    out = []
    for i in range(n_utts):
        if nh[i] < 0:
            out.append(None)
            continue
        out.append([([int(x) for x in words[i, j, :min(int(nw[i, j]), max_words)]], float(g[i, j]), float(a[i, j]))
                    for j in range(int(nh[i]))])
    return out


def _posteriors(n_arcs, n_utts, call, get):
    """Runs call(totals, n_post) and get(arc_posts, frame_entries) for n_utts utterances whose
    lattices have n_arcs records (or negative codes) and unpacks them as Batch.posteriors returns
    them."""
    tot = np.zeros(max(n_utts, 1), np.float64)
    npost = np.zeros(max(n_utts, 1), np.int64)
    _check(call(tot.ctypes.data, npost.ctypes.data))
    if len(n_arcs) != n_utts:
        raise PkbError(1, "posteriors: the record counts of the latest lattice() are unknown")
    npost = npost[:n_utts]
    arc = np.empty(max(int(np.maximum(n_arcs, 0).sum()), 1), np.float32)
    fr = np.empty(max(int(np.maximum(npost, 0).sum()), 1), FRAME_POST_DTYPE)
    _check(get(arc.ctypes.data, fr.ctypes.data))
    return tot[:n_utts].copy(), _split(arc, n_arcs), _split(fr, npost)


def _best_path(n_utts, call, get):
    """Runs call(costs, graph_costs, acoustic_costs, n_words, n_frames) and get(words, word_t, ali) for
    n_utts utterances and unpacks them as Batch.best_path returns them."""
    u = max(n_utts, 1)
    cost, g, a = (np.zeros(u, np.float64) for _ in range(3))
    nw = np.zeros(u, np.int32)
    nf = np.zeros(u, np.int32)
    _check(call(cost.ctypes.data, g.ctypes.data, a.ctypes.data, nw.ctypes.data, nf.ctypes.data))
    nw, nf = nw[:n_utts], nf[:n_utts]
    words = np.empty(max(int(np.maximum(nw, 0).sum()), 1), np.int32)
    word_t = np.empty_like(words)
    ali = np.empty(max(int(nf.sum()), 1), np.int32)
    _check(get(words.ctypes.data, word_t.ctypes.data, ali.ctypes.data))
    ws, ts, al = _split(words, nw), _split(word_t, nw), _split(ali, np.where(nw < 0, -1, nf))
    return [None if nw[i] < 0 else (float(cost[i]), float(g[i]), float(a[i]), ws[i], ts[i], al[i])
            for i in range(n_utts)]


class Stream:
    """pkb_stream_t: n_streams audio streams advancing in lock step with carried state
    (PCM tail, CMVN running sums + ring, splice context). No reference equivalent exists; the
    contract is: concatenated outputs == whole-utterance outputs."""

    def __init__(self, ctx, am, n_streams, chunk_samples, global_stats, prob_scale=1.0):
        self.ctx, self.am = ctx, am
        self.n_streams, self.chunk = n_streams, chunk_samples
        self.h = _VP()
        _check(ctx.lib.pkb_stream_create(ctx.h, am.h, n_streams, chunk_samples, _f32(global_stats),
                                         prob_scale, C.byref(self.h)))
        ctx._adopt(self)
        self.max_frames = ctx.lib.pkb_stream_max_frames(self.h)
        self.P = am.num_pdfs()
        self.out = np.empty((n_streams, self.max_frames, self.P), np.float32)

    def close(self):
        if self.h:
            self.ctx.lib.pkb_stream_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def push(self, pcm, out=None, rows=True):
        """pcm: int16 [n_streams][chunk]. Returns a view [n_streams][frames][P] (frames may be 0).
        rows=False (needs an attached decoder): no row is copied back; returns the frame count."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        assert pcm.shape == (self.n_streams, self.chunk)
        out = self.out if out is None else out
        n = C.c_int32(0)
        _check(self.ctx.lib.pkb_stream_push_i16(self.h, pcm.ctypes.data, out.ctypes.data if rows else None,
                                                C.byref(n)))
        return out[:, :n.value] if rows else n.value

    def flush(self, out=None, rows=True):
        out = self.out if out is None else out
        n = C.c_int32(0)
        _check(self.ctx.lib.pkb_stream_flush(self.h, out.ctypes.data if rows else None, C.byref(n)))
        return out[:, :n.value] if rows else n.value

    def graph_replays(self):
        """Pushes so far that replayed a captured CUDA graph (pkb_stream_graph_replays)."""
        n = C.c_int64(0)
        _check(self.ctx.lib.pkb_stream_graph_replays(self.h, C.byref(n)))
        return n.value

    def set_decoder(self, dec):
        """Attach a Decoder (None detaches): every push / flush advances it on the device."""
        _check(self.ctx.lib.pkb_stream_set_decoder(self.h, dec.h if dec is not None else None))
        self.decoder = dec

    def set_compact(self, on=True):
        """Half-size output rows (see pkb_stream_set_compact): push_compact / flush_compact."""
        _check(self.ctx.lib.pkb_stream_set_compact(self.h, 1 if on else 0))
        if on and not hasattr(self, "out16"):
            self.out16 = np.empty((self.n_streams, self.max_frames, self.P), np.uint16)
            self.out_off = np.empty((self.n_streams, self.max_frames), np.float32)

    def push_compact(self, pcm, out16=None, out_off=None):
        """Returns views (h16 [n_streams][frames][P], off [n_streams][frames])."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        assert pcm.shape == (self.n_streams, self.chunk)
        out16 = self.out16 if out16 is None else out16
        out_off = self.out_off if out_off is None else out_off
        n = C.c_int32(0)
        _check(self.ctx.lib.pkb_stream_push_compact_i16(self.h, pcm.ctypes.data, out16.ctypes.data,
                                                        out_off.ctypes.data, C.byref(n)))
        return out16[:, :n.value], out_off[:, :n.value]

    def flush_compact(self, out16=None, out_off=None):
        out16 = self.out16 if out16 is None else out16
        out_off = self.out_off if out_off is None else out_off
        n = C.c_int32(0)
        _check(self.ctx.lib.pkb_stream_flush_compact(self.h, out16.ctypes.data, out_off.ctypes.data, C.byref(n)))
        return out16[:, :n.value], out_off[:, :n.value]
