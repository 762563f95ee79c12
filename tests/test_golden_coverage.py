"""Every compiled (KIND, QT, D) instantiation of the fused kernels, the dense builder, the staged
engine and lg_predict (pgmuvi_b200/build.py CONFIGS) is reached by at least one golden case, so a
fault in any one of them fails the golden-parametrised GPU tests.  Runs without a GPU."""
from conftest import golden_names, load_golden
from pgmuvi_b200.build import CONFIGS

SEP_KINDS = (3, 4, 5, 6)
STAT_BASE = 8


def pad_q(Q):
    """csrc/cabi.cu pad_q: the mixture count rounded up to a compiled QT."""
    return 1 if Q <= 1 else 2 if Q <= 2 else 4 if Q <= 4 else 8


def instantiation(kind, Q, d):
    """(KIND, QT, D) that csrc/cabi.cu's PGM_DISPATCH sends a (kind, Q, d) model to."""
    if kind >= STAT_BASE:
        return (kind, 4, d)                      # stationary kinds: no mixtures, QT = 4
    if kind in SEP_KINDS:
        return (kind, 4 if Q <= 4 else 8, d)     # PGM_DISPATCH_Q48
    return (kind, pad_q(Q), d)


def _golden_instantiations():
    out = {}
    for name in golden_names():
        g = load_golden(name)
        out.setdefault(instantiation(g["kind"], g["Q"], g["d"]), []).append((name, g["Q"]))
    return out


def test_every_compiled_instantiation_has_a_golden():
    reached = _golden_instantiations()
    missing = sorted(c for c in CONFIGS if c not in reached)
    assert not missing, f"(KIND, QT, D) compiled but reached by no tests/golden case: {missing}"
    extra = sorted(c for c in reached if c not in CONFIGS)
    assert not extra, f"golden cases dispatch to instantiations that are not compiled: {extra}"


def test_padded_mixtures_of_qt8_are_covered():
    """Q = 5..7 runs QT = 8 with padded mixtures (what the flicker term produces at the default
    num_mixtures = 4); the one-block-per-SM ARD kind (1, 8, 2) is covered with all 8 mixtures."""
    reached = _golden_instantiations()
    gaps = []
    for c in CONFIGS:
        kind, qt, _ = c
        if qt != 8:
            continue
        qs = {Q for _, Q in reached.get(c, [])}
        want = {8} if c == (1, 8, 2) else {5, 6, 7}
        if not qs & want:
            gaps.append((c, sorted(qs)))
    assert not gaps, f"QT = 8 instantiations without a golden of the required Q: {gaps}"
