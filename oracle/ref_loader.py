"""ORACLE (test infrastructure) — import the REAL reference package from /root/reference.

Only usable where the reference tree exists; no test needs it.  Used by the fixture generators
tests/golden/make_golden*.py to pin the restatement in oracle/*.py against the reference's
own modules.  Nothing is copied: the reference is
imported in place through three stub packages (oracle/stubs) for its missing deps.
"""
import os
import sys

REF_ROOT = "/root/reference"
_STUBS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "stubs")


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "wesep"))


def import_reference():
    """Returns the reference `wesep` package (models importable) or raises RuntimeError."""
    if not available():
        raise RuntimeError("reference tree not present at " + REF_ROOT)
    for p in (REF_ROOT, _STUBS):
        if p not in sys.path:
            sys.path.insert(0, p)
    import wesep  # noqa: F401
    import wesep.models.convtasnet  # noqa: F401
    return wesep


SPEXPLUS_ARGS = dict(  # examples/librimix/tse/v2/confs/spexplus.yaml:36-56
    B=256, H=512, L=20, N=256, P=3, R=4, X=8, spk_emb_dim=256, activate="relu", causal=False, norm="gLN",
    skip_con=False, spk_fuse_type="concatConv", use_spk_transform=False, multi_fuse=True, encoder_type="Multi",
    decoder_type="Multi", joint_training=True, multi_task=True, spksInTrain=251)
