"""oracle/fetch_ref.py: the recipe that puts the UNMODIFIED reference under the git-ignored oracle/_ref/ (so that a copy of
the tree taken to a GPU machine carries it like a built .so) and imports it under private module names."""
import os
import subprocess
import sys

import pytest

from oracle import fetch_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ref_dir_is_git_ignored_but_travels():
    gi = open(os.path.join(ROOT, ".gitignore")).read()
    assert "oracle/_ref/" in gi
    gpi = os.path.join(ROOT, ".gpurunignore")
    assert not os.path.exists(gpi) or "oracle/_ref" not in open(gpi).read()
    tracked = subprocess.run(["git", "ls-files", "oracle/_ref"], cwd=ROOT, capture_output=True, text=True).stdout.strip()
    assert tracked == "", "reference sources must never be committed"


def test_fetch_copies_verbatim(tmp_path, monkeypatch):
    """The copy is byte for byte (CRLF, trailing whitespace, non-UTF-8 bytes survive) and verify() notices an edit.  Runs on
    a stand-in source tree so that it needs no checkout of the reference."""
    src, dst = tmp_path / "reference", tmp_path / "_ref"
    src.mkdir()
    for i, n in enumerate(fetch_ref.FILES):
        (src / n).write_bytes(b"# %s\r\nx = %d  \n\xff\xfe\n" % (n.encode(), i))
    monkeypatch.setattr(fetch_ref, "REF_SRC", str(src))
    monkeypatch.setattr(fetch_ref, "REF_DST", str(dst))
    assert fetch_ref.fetch(verbose=False)
    for n in fetch_ref.FILES:
        assert open(os.path.join(fetch_ref.REF_SRC, n), "rb").read() == open(os.path.join(fetch_ref.REF_DST, n), "rb").read()
    assert fetch_ref.available() and fetch_ref.verify()
    (dst / fetch_ref.FILES[0]).write_bytes(b"edited\n")
    assert not fetch_ref.verify()
    monkeypatch.setattr(fetch_ref, "REF_SRC", "")
    assert not fetch_ref.fetch(verbose=False)          # no reference tree given: nothing happens


def test_find_reference_env_then_sibling_checkout(tmp_path, monkeypatch):
    (tmp_path / "repo" / "oracle").mkdir(parents=True)
    monkeypatch.setattr(fetch_ref, "HERE", str(tmp_path / "repo" / "oracle"))
    monkeypatch.delenv("VAE_SONG_REFERENCE", raising=False)
    assert fetch_ref.find_reference() == ""
    (tmp_path / "vae-song").mkdir()
    (tmp_path / "vae-song" / "module.py").write_text("")
    assert fetch_ref.find_reference() == str(tmp_path / "vae-song")
    (tmp_path / "reference").mkdir()
    assert fetch_ref.find_reference() == str(tmp_path / "vae-song")          # a directory without module.py is not one
    (tmp_path / "reference" / "module.py").write_text("")
    assert fetch_ref.find_reference() == str(tmp_path / "reference")
    monkeypatch.setenv("VAE_SONG_REFERENCE", str(tmp_path / "elsewhere"))
    assert fetch_ref.find_reference() == str(tmp_path / "elsewhere")


@pytest.mark.skipif(not fetch_ref.available(), reason="oracle/_ref not populated")
def test_import_under_private_names_and_runs():
    import torch
    before = {n: sys.modules.get(n) for n in ("module", "model", "utils", "dataset", "lipschitz")}
    ns = fetch_ref.import_ref()
    assert {n: sys.modules.get(n) for n in before} == before            # nothing shadows vae_song_b200's modules
    assert ns.model.LIDVAE.__module__ == "_ref_model" and ns.lipschitz.train_model.__module__ == "_ref_lipschitz"
    torch.manual_seed(0)
    m = ns.model.LIDVAE(dataset="pinwheel", icnn_channels=[16, 32], hidden_channels=[8, 4])
    ns.lipschitz.train_model(m, [(torch.randn(32, 2), None)] * 2, epochs=1, lr=1e-3, device="cpu")
    assert all(torch.isfinite(p).all() for p in m.parameters())
