"""Import the UNMODIFIED reference code — TEST / BENCH INFRASTRUCTURE, never imported by the product package.

The reference is a checkout of the original project (iamwangyabin/hardnetNas), which this repository does not contain;
by default it is looked for next to the repository, at ../reference. `stage()` (run by __graft_entry__.build()) copies the
handful of reference files this hot path consists of, byte for byte, into oracle/_ref/ — a git-ignored directory that
travels with the tree like the built .so does — so that `bench.py --impl reference` and the cpu_baseline records time the
reference's own classes (cpu_baseline.kind = "reference"); without it they time the oracle port. Where the checkout is
missing or unreadable, staging is skipped. `python oracle/ref_loader.py <checkout>` stages from another location. Nothing
under oracle/_ref/ is ever committed, edited or read by hardnetnas_b200/.

The import recipes work around the reference's import-time side effects (SURVEY.md section 8c): hardnet/HardNet.py parses
argv, sets CUDA_VISIBLE_DEVICES and creates data/logs/ in the cwd; LookUpTable() reads a path relative to hardnetNAS/.
"""
from __future__ import annotations

import os
import shutil
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
REFERENCE = HERE.parent.parent / "reference"
STAGED = HERE / "_ref"

# relative paths of the files the hot path consists of (SURVEY.md section 8a)
FILES = [
    "hardnet/HardNet.py", "hardnet/Losses.py", "hardnet/Utils.py", "hardnet/EvalMetrics.py",
    "FDLNet-master/utils/eval_utils.py", "FDLNet-master/utils/math_utils.py",
    "hardnetNAS/fbnet_building_blocks/fbnet_builder.py", "hardnetNAS/fbnet_building_blocks/fbnet_modeldef.py",
    "hardnetNAS/fbnet_building_blocks/layers/__init__.py", "hardnetNAS/fbnet_building_blocks/layers/batch_norm.py",
    "hardnetNAS/fbnet_building_blocks/layers/misc.py",
    "hardnetNAS/supernet_functions/lookup_table_builder.py", "hardnetNAS/supernet_functions/lookup_table.txt",
    "hardnetNAS/supernet_functions/config_for_supernet.py", "hardnetNAS/general_functions/utils.py",
]


def _complete(tree: Path) -> bool:
    """Every file of FILES is under `tree`. A tree the user may not read counts as absent (Path.exists() raises
    PermissionError there instead of returning False)."""
    try:
        return all((tree / rel).is_file() for rel in FILES)
    except OSError:
        return False


def stage(source: Path | None = None, dest: Path = STAGED) -> Path | None:
    """Copy the reference files of the checkout `source` (default REFERENCE) into `dest`. Where the source is missing or
    unreadable nothing is copied. Returns `dest` if it holds a complete copy afterwards, else None."""
    source = REFERENCE if source is None else Path(source)
    if _complete(source):
        try:
            for rel in FILES:
                dst = dest / rel
                dst.parent.mkdir(parents=True, exist_ok=True)
                shutil.copyfile(source / rel, dst)
        except OSError as exc:
            print(f"[ref_loader] staging the reference from {source} failed: {exc}", file=sys.stderr)
    return dest if _complete(dest) else None


def root() -> Path | None:
    """Where the reference can be imported from: the checkout if present, else the staged copy, else None."""
    for tree in (REFERENCE, STAGED):
        if _complete(tree):
            return tree
    return None


def load_hardnet(ref: Path | None = None):
    """(HardNet module, Losses module, EvalMetrics module) of hardnet/."""
    ref = ref or root()
    if ref is None:
        raise FileNotFoundError(f"reference sources are neither at {REFERENCE} nor staged under oracle/_ref")
    saved_argv, saved_cwd = sys.argv, os.getcwd()
    saved_env = os.environ.get("CUDA_VISIBLE_DEVICES")
    tmp = tempfile.mkdtemp(prefix="hn_ref_")
    os.chdir(tmp)
    sys.argv = ["HardNet.py"]
    sys.path.insert(0, str(ref / "hardnet"))
    try:
        import HardNet as ref_hardnet  # noqa: N813
        import Losses as ref_losses
        import EvalMetrics as ref_metrics
    finally:
        sys.argv = saved_argv
        os.chdir(saved_cwd)
        sys.path.remove(str(ref / "hardnet"))
        if saved_env is None:
            os.environ.pop("CUDA_VISIBLE_DEVICES", None)
        else:
            os.environ["CUDA_VISIBLE_DEVICES"] = saved_env
        shutil.rmtree(tmp, ignore_errors=True)
    return ref_hardnet, ref_losses, ref_metrics


def load_fdl(ref: Path | None = None):
    """(eval_utils, math_utils) of FDLNet-master/utils."""
    ref = ref or root()
    if ref is None:
        raise FileNotFoundError(f"reference sources are neither at {REFERENCE} nor staged under oracle/_ref")
    for m in [k for k in sys.modules if k == "utils" or k.startswith("utils.")]:
        del sys.modules[m]
    sys.path.insert(0, str(ref / "FDLNet-master"))
    try:
        from utils import eval_utils, math_utils
    finally:
        sys.path.remove(str(ref / "FDLNet-master"))
    return eval_utils, math_utils


def load_nas(ref: Path | None = None):
    """(PRIMITIVES, ConvBNRelu, Flatten, LookUpTable instance) of hardnetNAS/."""
    ref = ref or root()
    if ref is None:
        raise FileNotFoundError(f"reference sources are neither at {REFERENCE} nor staged under oracle/_ref")
    nas = ref / "hardnetNAS"
    cwd = os.getcwd()
    os.chdir(nas)   # LookUpTable() reads ./supernet_functions/lookup_table.txt
    sys.path.insert(0, str(nas))
    for m in [k for k in sys.modules if k.split(".")[0] in ("fbnet_building_blocks", "supernet_functions", "general_functions")]:
        del sys.modules[m]
    try:
        from fbnet_building_blocks.fbnet_builder import PRIMITIVES, ConvBNRelu, Flatten
        from supernet_functions.lookup_table_builder import LookUpTable
        table = LookUpTable()
    finally:
        os.chdir(cwd)
        sys.path.remove(str(nas))
    return PRIMITIVES, ConvBNRelu, Flatten, table


if __name__ == "__main__":
    if len(sys.argv) > 2:
        raise SystemExit("usage: python oracle/ref_loader.py [checkout of the original hardnetNas project, default ../reference]")
    print(stage(Path(sys.argv[1]) if len(sys.argv) == 2 else None))
