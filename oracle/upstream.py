"""The upstream speech-to-speech package (huggingface/speech-to-speech) for the tests of the drop-in boundary -- TEST
INFRASTRUCTURE ONLY.

Those tests check that our handlers subclass the upstream base classes, register in its backend registry and run its request
lifecycle.  `build()` byte-compiles the `speech_to_speech` package of an upstream checkout into oracle/_ref/ (a build product,
kept out of git), so the tests import it from this tree; `importable()` puts it on sys.path.  The checkout's src/ directory is
taken from $S2S_UPSTREAM_SRC, else from /root/reference/src, where the build machines keep it.  Without a checkout nothing is
staged, an installed `speech_to_speech` is used if there is one, and otherwise those tests skip.
"""
from __future__ import annotations

import importlib.util
import os
import py_compile
import shutil
import sys

REF_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
PACKAGE = "speech_to_speech"


def source_dir() -> str | None:
    src = os.environ.get("S2S_UPSTREAM_SRC") or "/root/reference/src"
    return src if os.path.isfile(os.path.join(src, PACKAGE, "__init__.py")) else None


def build() -> bool:
    """Stage the upstream package as sourceless bytecode under oracle/_ref/ (rebuilt every time); False without a checkout."""
    src = source_dir()
    if src is None:
        return False
    dest = os.path.join(REF_DIR, PACKAGE)
    shutil.rmtree(dest, ignore_errors=True)
    for root, dirs, files in os.walk(os.path.join(src, PACKAGE)):
        dirs[:] = [d for d in dirs if d != "__pycache__"]
        rel = os.path.relpath(root, src)
        for f in files:
            if f.endswith(".py"):
                py_compile.compile(os.path.join(root, f), cfile=os.path.join(REF_DIR, rel, f + "c"),
                                   dfile=os.path.join(rel, f), doraise=True)
    return True


def importable() -> bool:
    """True when `import speech_to_speech` works: the staged copy (put first on sys.path) or an installed package."""
    if os.path.isfile(os.path.join(REF_DIR, PACKAGE, "__init__.pyc")) and REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    return importlib.util.find_spec(PACKAGE) is not None
