"""CPU: the drop-in boundary (SURVEY §8b) — registry names, call conventions, and INTEGRATION.md option (ii) against
registry modules laid out like the reference's."""
import inspect
import sys

import pytest


def test_registries_hold_the_reference_names():
    from ctdd_b200.lib.sampling import sampling_utils as su
    from ctdd_b200.lib.losses import losses_utils as lu
    import ctdd_b200.lib.sampling.sampling  # noqa: F401
    import ctdd_b200.lib.losses.losses  # noqa: F401
    for name in ("TauL", "LBJF", "MidPointTauL", "PCTauL", "ConditionalTauLeaping", "ConditionalPCTauLeaping", "ExactSampling"):
        assert name in su._SAMPLERS, name
    for name in ("CTElbo", "NLL", "CTElboLambda", "CondCTElbo", "CatRM", "CatRMNLL", "ScoreElbo", "SDDMElbo", "NLLOriginal"):
        assert name in lu._LOSSES, name
    with pytest.raises(ValueError):                 # duplicate registration is an error, as in the reference
        su.register_sampler(su._SAMPLERS["TauL"])
    with pytest.raises(ValueError):
        lu.register_loss(lu._LOSSES["CTElbo"])


def test_sampler_and_loss_signatures_match_the_reference_conventions():
    from ctdd_b200.lib.sampling import sampling as s
    from ctdd_b200.lib.losses import losses as l
    assert list(inspect.signature(s.TauL.sample).parameters) == ["self", "model", "N"]
    assert list(inspect.signature(s.ConditionalTauLeaping.sample).parameters) == ["self", "model", "N", "conditioner"]
    assert list(inspect.signature(s.get_initial_samples).parameters)[:6] == ["N", "D", "device", "S", "initial_dist", "initial_dist_std"]
    for cls in (l.CTElbo, l.CatRM, l.SDDMElbo, l.ScoreElbo, l.CatRMNLL, l.NLLOriginal):
        assert len(inspect.signature(cls.calc_loss).parameters) >= 3     # (self, a, b[, label/writer]): both orders accepted


def test_no_cpu_fallback_is_offered():
    """Host tensors are refused instead of being routed to a CPU path."""
    import torch
    from ctdd_b200 import _native as nat
    with pytest.raises(RuntimeError):
        nat.ptr(torch.zeros(4))


_REGISTRY = """\
TABLE = {}


def register_KIND(cls):
    if cls.__name__ in TABLE:
        raise ValueError(cls.__name__ + " is already registered!")
    TABLE[cls.__name__] = cls
    return cls


def get_KIND(cfg):
    return TABLE[cfg.KIND.name](cfg)
"""


def test_install_into_reference_overwrites_the_reference_registries(tmp_path, monkeypatch):
    """A train script has imported the reference's `lib.sampling.sampling` / `lib.losses.losses`: after
    install_into_reference() its registries resolve to our classes.  The reference's modules are stood in for by modules
    at the same import paths, written independently of ours: a module-level name -> class dict filled by a
    decorator that refuses duplicates, each registering one class of its own."""
    import ctdd_b200
    from ctdd_b200.lib.sampling import sampling as ours, sampling_utils as our_su
    from ctdd_b200.lib.losses import losses_utils as our_lu
    for pkg, table, kind, cls in (("sampling", "_SAMPLERS", "sampler", "TauL"), ("losses", "_LOSSES", "loss", "CTElbo")):
        d = tmp_path / "lib" / pkg
        d.mkdir(parents=True)
        (d / "__init__.py").write_text("")
        (d / f"{pkg}_utils.py").write_text(_REGISTRY.replace("TABLE", table).replace("KIND", kind))
        (d / f"{pkg}.py").write_text(f"from lib.{pkg}.{pkg}_utils import register_{kind}\n\n\n"
                                     f"@register_{kind}\nclass {cls}:\n    pass\n")
    (tmp_path / "lib" / "__init__.py").write_text("")
    monkeypatch.syspath_prepend(str(tmp_path))
    is_lib = lambda m: m == "lib" or m.startswith("lib.")
    for m in [m for m in sys.modules if is_lib(m)]:
        monkeypatch.delitem(sys.modules, m)
    try:
        import lib.sampling.sampling as rs
        import lib.losses.losses as rl
        import lib.sampling.sampling_utils as ref_su
        import lib.losses.losses_utils as ref_lu
        assert ref_su is not our_su and ref_lu is not our_lu
        before = ref_su._SAMPLERS["TauL"]
        assert before is rs.TauL and ref_lu._LOSSES["CTElbo"] is rl.CTElbo
        samplers, losses = ctdd_b200.install_into_reference()
        assert ref_su._SAMPLERS["TauL"] is ours.TauL and ref_su._SAMPLERS["TauL"] is not before
        assert "CTElbo" in losses and ref_lu._LOSSES["CTElbo"].__module__.startswith("ctdd_b200")
        assert sorted(ref_su._SAMPLERS) == samplers and sorted(ref_lu._LOSSES) == losses
    finally:
        for m in [m for m in sys.modules if is_lib(m)]:
            del sys.modules[m]


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver times next to ours) writes exactly one JSON line to stdout,
    carrying the metric / unit / config of our arm plus cpu_baseline and a zero-copy e2e block."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "reverse_step_tflops" and d["unit"] == "TFLOP/s"
    assert d["higher_is_better"] is True and d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["value"] > 0

