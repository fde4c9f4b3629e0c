#!/usr/bin/env python
"""Populate oracle/_ref/ with the UNMODIFIED reference (test / baseline infrastructure, not product code).

    python oracle/fetch_ref.py       # reference: $VAE_SONG_REFERENCE, else ../reference or ../vae-song beside the repo

The reference is a set of Python scripts without packaging (nothing to `pip install`), and the repository does not ship
it: it is taken from $VAE_SONG_REFERENCE or, without that, from a checkout named `reference` or `vae-song` in the
directory that holds this repository (`find_reference()`; build() runs `fetch()`).  This recipe copies the reference's own files for the hot path -- module.py, model.py, utils.py, lipschitz.py,
dataset.py -- byte for byte into the git-ignored oracle/_ref/ (so that a copy of the tree taken to a GPU machine carries
them like a built .so), plus SHA-256 digests in oracle/_ref/MANIFEST.json.  Nothing under
oracle/_ref/ is ever committed, and the product package never imports it (tests/test_abi_host_cpu.py enforces that).

`import_ref()` is how tests/, bench.py's reference arm and __graft_entry__.smoke() reach it: utils.py / lipschitz.py import
matplotlib (absent from the image) at module scope, so empty stub modules are registered first (SURVEY.md 8(c)); the
reference modules are loaded under PRIVATE names (`_ref_module`, `_ref_model`, ...) with `module` / `model` / `utils` /
`dataset` bound in sys.modules only while they import one another, so they never shadow vae_song_b200's modules.
"""
from __future__ import annotations

import hashlib
import importlib.util
import json
import os
import shutil
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
SIBLINGS = ("reference", "vae-song")       # checkout names looked for beside the repository


def find_reference() -> str:
    """Directory of the unmodified reference: $VAE_SONG_REFERENCE if set, else the first sibling checkout of this
    repository in SIBLINGS that has the reference's module.py; "" when there is none."""
    env = os.environ.get("VAE_SONG_REFERENCE")
    if env:
        return env
    parent = os.path.dirname(os.path.dirname(HERE))
    for name in SIBLINGS:
        if os.path.isfile(os.path.join(parent, name, "module.py")):
            return os.path.join(parent, name)
    return ""


REF_SRC = find_reference()
REF_DST = os.path.join(HERE, "_ref")
FILES = ("module.py", "model.py", "utils.py", "lipschitz.py", "dataset.py")


def _sha(path):
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()


def fetch(verbose=True) -> bool:
    """Copy FILES verbatim from the reference tree.  Returns False (and leaves _ref/ alone) when the tree is absent."""
    if not (REF_SRC and os.path.isdir(REF_SRC)):
        if verbose:
            print(f"fetch_ref: no reference checkout (VAE_SONG_REFERENCE unset, no {' or '.join('../' + s for s in SIBLINGS)} "
                  f"beside the repository); keeping {REF_DST} as it is")
        return False
    os.makedirs(REF_DST, exist_ok=True)
    manifest = {}
    for name in FILES:
        src, dst = os.path.join(REF_SRC, name), os.path.join(REF_DST, name)
        shutil.copyfile(src, dst)
        os.chmod(dst, 0o644)
        manifest[name] = _sha(dst)
        assert manifest[name] == _sha(src)
    with open(os.path.join(REF_DST, "MANIFEST.json"), "w") as f:
        json.dump({"source": REF_SRC, "sha256": manifest}, f, indent=1)
    if verbose:
        print(f"fetch_ref: {len(FILES)} reference files -> {REF_DST}")
    return True


def available() -> bool:
    return all(os.path.exists(os.path.join(REF_DST, n)) for n in FILES)


def verify() -> bool:
    """True when every file under _ref/ still has the digest recorded at fetch time (i.e. it is unmodified)."""
    try:
        man = json.load(open(os.path.join(REF_DST, "MANIFEST.json")))["sha256"]
        return all(_sha(os.path.join(REF_DST, n)) == man[n] for n in FILES)
    except Exception:
        return False


_cache = {}


def import_ref(swap=None):
    """Import the unmodified reference from oracle/_ref/ and return a namespace with .module .model .utils .dataset
    .lipschitz.

    swap: optional {"module": mod, "model": mod, "utils": mod} -- modules bound under those names INSTEAD of the
    reference's while `lipschitz.py` imports them: the drop-in test (the reference's own driver file running on
    vae_song_b200's classes).  Swapped imports are not cached."""
    key = None if not swap else tuple(sorted(swap))
    if key is None and "ns" in _cache:
        return _cache["ns"]
    if not available():
        raise FileNotFoundError(f"{REF_DST} is not populated: run `python oracle/fetch_ref.py` where a reference checkout is found")
    for name in ("matplotlib", "matplotlib.pyplot"):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib"].use = getattr(sys.modules["matplotlib"], "use", lambda *a, **k: None)

    public = ("module", "model", "utils", "dataset", "lipschitz")
    saved = {n: sys.modules.get(n) for n in public}
    ns = types.SimpleNamespace()
    try:
        for n in public:
            sys.modules.pop(n, None)
        for n in ("module", "model", "utils", "dataset", "lipschitz"):
            if swap and n in swap:
                mod = swap[n]
            else:
                spec = importlib.util.spec_from_file_location(f"_ref_{n}", os.path.join(REF_DST, f"{n}.py"))
                mod = importlib.util.module_from_spec(spec)
                sys.modules[n] = mod              # visible to the reference's own `import module` / `from model import ...`
                spec.loader.exec_module(mod)
                sys.modules[f"_ref_{n}"] = mod
            sys.modules[n] = mod
            setattr(ns, n, mod)
    finally:
        for n in public:
            if saved[n] is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = saved[n]
    if key is None:
        _cache["ns"] = ns
    return ns


if __name__ == "__main__":
    ok = fetch()
    sys.exit(0 if ok else 1)
