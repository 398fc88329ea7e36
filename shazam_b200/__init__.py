"""sia-b200: B200-native fingerprint-and-match path of SIA (CarlosArturoMe/shazam).

Layout (only what the hot path needs):
  csrc/            sm_100a CUDA kernels + the C ABI (include/sia_b200.h)
  _native.py       ctypes binding of the C ABI — no CPU fallback
  fingerprinter.py array-typed host driver (K1 STFT->dB, K2 peaks, K3 pairs+SHA-1)
  compat.py        the reference's function names/signatures on top of it
  stream.py        StreamFingerprinter: many concurrent streams fed block by block, same hashes as whole tracks
"""
__version__ = "0.1.0"

from . import _native  # noqa: F401


def __getattr__(name):
    # torch-dependent modules are imported lazily so that `import shazam_b200` stays cheap
    if name in ("Fingerprinter", "FingerprintBatch", "pack_tracks", "digests_to_hex", "hex_to_digests",
                "as_pcm_int16"):
        from . import fingerprinter
        return getattr(fingerprinter, name)
    if name in ("compat", "fingerprinter", "database", "recognize", "distributed", "stream"):
        import importlib
        return importlib.import_module(f"{__name__}.{name}")
    raise AttributeError(name)
