"""pocketkaldi_b200 -- B200-native (sm_100a) acoustic front half of pocketkaldi.

The product is the C-ABI library `libpkb200.so` (include/pkb200.h) built from
pocketkaldi_b200/csrc. This package is the Python host binding used by the tests and
bench.py; it mirrors the reference's C++ interfaces for this path (`Fbank`, `CMVN`,
`Nnet`, `AcousticModel`, `Decodable`, same method names and argument meaning) on top
of that ABI. There is no CPU fallback: importing works anywhere (so CPU-only tests can
check symbols), but every compute call needs the CUDA library and an sm_100 device and
raises `PkbError` otherwise.
"""

from .binding import (  # noqa: F401
    LIB_PATH,
    PkbError,
    Context,
    Fbank,
    CMVN,
    Nnet,
    AcousticModel,
    Decodable,
    Event,
    Batch,
    Decoder,
    Fst,
    LATTICE_ARC_DTYPE,
    FRAME_POST_DTYPE,
    Stream,
    WavList,
    read_wav,
    build_library,
    load_library,
    PREC_BF16,
    PREC_BF16X3,
    PREC_FP16,
    PREC_FP16X3,
    PREC_FP16C8,
    PREC_FP16R,
    STAGE_FBANK,
    STAGE_CMVN,
    STAGE_NNET,
    STAGE_ALL,
    STAGE_NO_FEATS,
    BUF_PCM,
    BUF_RAW,
    BUF_FEATS,
    BUF_LOGLIK,
    BUF_LOGLIK16,
    BUF_LOGLIK_OFF,
    KERNEL_CLASSES,
)
