"""Vendoring recipe for the reference arm — TEST / BENCH INFRASTRUCTURE, not product code.

The reference (Roestlab/diffusion-deconvolution-dia-msms-data) is pure Python: there is nothing to compile.  This
script copies the UNMODIFIED modules of the hot path from a checkout of the reference into oracle/_ref/ (git-ignored)
together with the two import shims the reference needs (rotary_embedding_torch: restated third-party arithmetic,
SURVEY.md §8c; duckdb: import-only, the .npy path never calls it).  `bench.py --impl reference` then times the
reference's own `DDIMDiffusionModel._train_one_batch` on the host cores (`cpu_baseline.kind = "reference"`), and
`bench.py` reports the same code on the B200 in eager fp32 as `gpu_eager_baseline`.

    python oracle/make_ref.py [CHECKOUT [DEST]]   # (re)creates DEST (default oracle/_ref/) from CHECKOUT
    DQUARTIC_REFERENCE=CHECKOUT python oracle/make_ref.py

CHECKOUT is the reference repository's root (the directory that holds `dquartic/`).  Without an argument or
DQUARTIC_REFERENCE the checkout at the default location (SRC below) is used; if that is absent, the script is a no-op
with exit 0 and oracle/_ref keeps whatever it holds.  A checkout that is named but missing is an error.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = "/root/reference/dquartic"
DST = os.path.join(HERE, "_ref")
FILES = ["model/model.py", "model/model_interface.py", "model/unet1d.py", "model/building_blocks.py",
         "utils/data_loader.py"]


def checkout(argv=()):
    """(root of the reference checkout, whether it was named explicitly): argv, else DQUARTIC_REFERENCE, else the
    default location."""
    named = argv[0] if argv else os.environ.get("DQUARTIC_REFERENCE")
    return (named, True) if named else (os.path.dirname(SRC), False)


def main(argv):
    root, named = checkout(argv)
    src = os.path.join(root, "dquartic")
    dst = argv[1] if len(argv) > 1 else DST
    if not os.path.isdir(src):
        if named:
            print(f"make_ref: {src} is not a directory", file=sys.stderr)
            return 1
        print(f"make_ref: {src} not present - keeping whatever oracle/_ref holds")
        return 0
    pkg = os.path.join(dst, "dquartic")
    if os.path.isdir(dst):
        shutil.rmtree(dst)
    for rel in FILES:
        out = os.path.join(pkg, rel)
        os.makedirs(os.path.dirname(out), exist_ok=True)
        shutil.copyfile(os.path.join(src, rel), out)
    # package markers written here (the reference's own __init__ imports cli / data_generation, which need polars etc.)
    for d in ("", "model", "utils"):
        open(os.path.join(pkg, d, "__init__.py"), "w").close()
    for shim in ("rotary_embedding_torch.py", "duckdb.py"):
        shutil.copyfile(os.path.join(HERE, "_shims", shim), os.path.join(dst, shim))
    print(f"make_ref: vendored {len(FILES)} reference modules into {dst}")
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
