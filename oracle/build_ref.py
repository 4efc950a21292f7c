"""TEST / BASELINE INFRASTRUCTURE -- vendors the UNMODIFIED reference hot-path files into oracle/_ref/.

    python oracle/build_ref.py        (also run by __graft_entry__.build() when /root/reference exists)

`oracle/_ref/` is a build output: git-ignored (reference sources never enter the history).  Where it exists it serves as
the CPU baseline of `bench.py` (`cpu_baseline.kind = "reference"`, `bench.py --impl reference`): the reference's own
`full_attention_conv` timed on the host cores; without it `bench.py` times the oracle's op-for-op port of that function
(`tests/test_oracle_golden.py` checks that the port runs the reference's op chain).
The files are byte-for-byte copies (checked below); they import under `oracle/ref_shim.py`, which stands in for the
three names of torch_sparse / torch_geometric the reference needs and this image lacks.
"""
import filecmp
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.environ.get("DIFFORMER_REFERENCE_SRC", "/root/reference")
DST = os.path.join(HERE, "_ref")
FILES = [os.path.join("node classification", "difformer.py"), os.path.join("physical particle", "difformer-v2.py")]


def build_ref(verbose: bool = True) -> bool:
    """Copy the reference files; returns False (and leaves any earlier copy in place) when the source tree is absent."""
    if not os.path.isfile(os.path.join(SRC, FILES[0])):
        if verbose:
            print(f"oracle/build_ref: {SRC} not present -- keeping whatever is in {DST}", file=sys.stderr)
        return False
    for rel in FILES:
        dst = os.path.join(DST, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(os.path.join(SRC, rel), dst)
        assert filecmp.cmp(os.path.join(SRC, rel), dst, shallow=False), f"copy of {rel} differs"
    if verbose:
        print(f"oracle/build_ref: {len(FILES)} reference files -> {DST}")
    return True


if __name__ == "__main__":
    sys.exit(0 if build_ref() else 1)
