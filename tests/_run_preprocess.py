#!/usr/bin/env python3
"""Runs the UNMODIFIED data_preprocess.py of a staged reference tree as ``__main__`` (test infrastructure).

    python tests/_run_preprocess.py --ref baseline/_ref --work WORKDIR

The environment shims are tests/_run_caller.py's (PyYAML loader, librosa stub with core.stft / filters.mel from
oracle/frontend.py), plus the two librosa calls data_preprocess.py adds: ``core.load`` (the float32 samples stored in
``path`` as .npy bytes, at the requested rate) and ``effects.split`` (tests/_preprocess_oracle.py's restatement of
librosa 0.6).  CWD = WORKDIR holds config/config.yaml and the speaker folders the config names.
"""
import argparse
import os
import runpy
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)


def install_shims():
    import numpy as np

    import _preprocess_oracle as P
    import _run_caller
    _run_caller.install_shims()
    librosa = sys.modules["librosa"]

    def load(path, sr=22050):
        return np.load(path, allow_pickle=False).astype(np.float32), sr

    librosa.core.load = load
    librosa.effects = types.ModuleType("librosa.effects")
    librosa.effects.split = lambda y, top_db=60: P.split(y, top_db)
    sys.modules["librosa.effects"] = librosa.effects


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", required=True)
    ap.add_argument("--work", required=True)
    a = ap.parse_args()
    ref = os.path.abspath(a.ref)
    install_shims()
    os.chdir(a.work)
    sys.path.insert(0, ref)
    runpy.run_path(os.path.join(ref, "data_preprocess.py"), run_name="__main__")
    print("PREPROCESS_OK")


if __name__ == "__main__":
    main()
