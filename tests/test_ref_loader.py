"""oracle/ref_loader.py: build() stages the original project's files into oracle/_ref/. A complete checkout is copied byte for
byte; a missing, incomplete or unreadable one is skipped without failing the build."""
import pathlib

from oracle import ref_loader


def _checkout(tmp_path):
    src = tmp_path / "reference"
    for i, rel in enumerate(ref_loader.FILES):
        f = src / rel
        f.parent.mkdir(parents=True, exist_ok=True)
        f.write_bytes(f"# reference file {i}\n".encode())
    return src


def test_stage_copies_a_complete_checkout_and_root_finds_it(tmp_path, monkeypatch):
    src = _checkout(tmp_path)
    dest = tmp_path / "_ref"
    assert ref_loader.stage(src, dest) == dest
    for rel in ref_loader.FILES:
        assert (dest / rel).read_bytes() == (src / rel).read_bytes()
    monkeypatch.setattr(ref_loader, "STAGED", dest)
    monkeypatch.setattr(ref_loader, "REFERENCE", src)
    assert ref_loader.root() == src                      # the checkout itself first
    monkeypatch.setattr(ref_loader, "REFERENCE", tmp_path / "absent")
    assert ref_loader.root() == dest                     # else the staged copy


def test_stage_skips_a_missing_or_incomplete_checkout(tmp_path):
    dest = tmp_path / "_ref"
    assert ref_loader.stage(tmp_path / "absent", dest) is None
    src = _checkout(tmp_path)
    (src / ref_loader.FILES[-1]).unlink()
    assert ref_loader.stage(src, dest) is None and not dest.exists()


def test_stage_and_root_skip_an_unreadable_checkout(tmp_path, monkeypatch):
    """Below a directory the user may not search, Path.is_file() raises PermissionError instead of returning False."""
    src = _checkout(tmp_path)
    dest = tmp_path / "_ref"
    real_is_file = pathlib.Path.is_file

    def is_file(self, *args, **kwargs):
        if src in self.parents:
            raise PermissionError(13, "Permission denied", str(self))
        return real_is_file(self, *args, **kwargs)
    monkeypatch.setattr(pathlib.Path, "is_file", is_file)
    assert ref_loader.stage(src, dest) is None and not dest.exists()
    monkeypatch.setattr(ref_loader, "REFERENCE", src)
    monkeypatch.setattr(ref_loader, "STAGED", dest)
    assert ref_loader.root() is None
