"""Resampler: the oracle against the reference's own compiled executor
(oracle/_ref), the library's designed filters against the oracle's, and the
reference's known-answer tests replayed on the oracle.  CPU only."""
import numpy as np
import pytest

from oracle import ref_executor, resample_oracle as R

RATE_PAIRS = [(44100, 48000), (48000, 44100), (44100, 16000), (16000, 44100), (44100, 22050),
              (22050, 44100), (48000, 8000), (8000, 48000), (3, 2)]

# oracle/_ref/libsoundml_ref.so is the reference SoundML's own C resampler, which oracle/Makefile
# compiles only from a checkout of the reference's source; that source is not part of this
# repository and no stored output of it exists, so without it these comparisons do not run.
needs_ref = pytest.mark.skipif(
    not ref_executor.available(),
    reason="needs oracle/_ref/libsoundml_ref.so, built only from the reference SoundML's C source "
           "(not in this repository)")


def oracle_stages(cfg):
    """Stage dicts for the oracle, every prototype designed by the oracle itself
    from the plan's (l, k, fc, beta)."""
    out = []
    for s in cfg.stages():
        out.append(dict(l=s["l"], m=s["m"], k=s["k"],
                        proto=R.design_prototype(s["l"], s["k"], s["fc"], s["beta"])))
    return out


@needs_ref
@pytest.mark.parametrize("sr,target", [(44100, 48000), (48000, 44100), (44100, 16000),
                                       (44100, 22050), (22050, 44100), (3, 2)])
def test_oracle_matches_reference_executor(sr, target):
    d = R.single_stage_design(sr, target)
    h = R.design_prototype(d["l"], d["k"], d["fc"], d["beta"])
    bank = R.bank_of_prototype(d["l"], d["k"], h)
    rng = np.random.default_rng(sr + target)
    for n in (1, 7, 500, 3000):
        x = rng.uniform(-1, 1, (2, n))
        total = R.ceil_div(n * d["l"], d["m"])
        want = R.stage_apply(x, h, d["l"], d["m"], d["k"], total)
        got64 = ref_executor.apply_single(x, bank, d["l"], d["m"], d["k"])
        assert got64.shape == want.shape
        peak = max(np.abs(want).max(), 1e-300)
        assert np.abs(got64 - want).max() / peak <= 1e-13
        got32 = ref_executor.apply_single(x.astype(np.float32), bank, d["l"], d["m"], d["k"])
        # the reference gates its own float32 surfaces at 32 units of peak * 2^-23
        assert np.abs(got32 - want).max() / peak <= 32 * 2.0 ** -23


@needs_ref
def test_oracle_cascade_matches_reference_executor(lib):
    cfg = lib.Resample.Config.create(sample_rate=48000, target=8000)
    st = oracle_stages(cfg)
    rng = np.random.default_rng(5)
    x = rng.uniform(-1, 1, (1, 4000))
    want = R.apply_plan(x, st, cfg.l, cfg.m)
    banks = [(R.bank_of_prototype(s["l"], s["k"], s["proto"]), s["l"], s["m"], s["k"]) for s in st]
    got = ref_executor.apply_cascade(x, banks[0], banks[1], cfg.l, cfg.m)
    assert got.shape == want.shape == (1, 667)
    assert np.abs(got - want).max() / np.abs(want).max() <= 1e-13


@pytest.mark.parametrize("sr,target", RATE_PAIRS)
def test_library_prototypes_match_oracle_design(lib, sr, target):
    cfg = lib.Resample.Config.create(sample_rate=sr, target=target)
    for i, s in enumerate(cfg.stages()):
        want = R.design_prototype(s["l"], s["k"], s["fc"], s["beta"])
        got = cfg.stage_prototype(i)
        assert got.shape == want.shape == (2 * s["k"] * s["l"] + 1,)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-18)
        assert abs(got.sum() - s["l"]) <= 1e-9 * s["l"]          # gain-normalised to L
        assert np.array_equal(got, got[::-1])                     # exact symmetry


def test_single_stage_design_matches_planner(lib):
    for sr, target in [(44100, 48000), (44100, 16000), (44100, 22050)]:
        cfg = lib.Resample.Config.create(sample_rate=sr, target=target)
        (s,) = cfg.stages()
        d = R.single_stage_design(sr, target)
        assert (s["l"], s["m"], s["k"]) == (d["l"], d["m"], d["k"])
        assert s["fc"] == d["fc"] and s["beta"] == d["beta"]
    # tier ladder K = 74 / 95 / 134 for 44.1 -> 48 kHz (resample_config.ml:46)
    for quality, k in (("fast", 74), ("high", 95), ("best", 134)):
        assert lib.Resample.Config.create(sample_rate=44100, target=48000, quality=quality).latency == k


# soundml/test/resample/resample_kernel.ml:99-109 — an impulse lands at j*L/M
@pytest.mark.parametrize("sr,target,quality,j,expected", [
    (44100, 48000, "high", 294, 320), (44100, 48000, "fast", 588, 640),
    (48000, 44100, "high", 320, 294), (44100, 22050, "high", 500, 250),
    (22050, 44100, "best", 250, 500), (44100, 16000, "high", 882, 320),
    (16000, 44100, "high", 320, 882), (48000, 8000, "high", 600, 100),
    (8000, 48000, "high", 100, 600)])
def test_impulse_lands_where_the_reference_says(lib, sr, target, quality, j, expected):
    cfg = lib.Resample.Config.create(sample_rate=sr, target=target, quality=quality)
    x = np.zeros(1000)
    x[j] = 1.0
    y = R.apply_plan(x, oracle_stages(cfg), cfg.l, cfg.m)
    assert int(np.argmax(np.abs(y))) == expected


def test_dc_is_alive_at_sample_zero(lib):
    cfg = lib.Resample.Config.create(sample_rate=44100, target=48000)
    y = R.apply_plan(np.ones(500), oracle_stages(cfg), cfg.l, cfg.m)
    assert 0.4 < y[0] < 1.05 and abs(y[200] - 1.0) < 1e-6


OLS_PAIRS = [(44100, 22050), (22050, 44100), (48000, 8000), (8000, 48000),
             (32000, 16000), (96000, 48000), (16000, 48000)]


@pytest.mark.parametrize("sr,target", OLS_PAIRS)
def test_planner_ols_geometry_matches_the_reference_rule(lib, sr, target):
    """The planner's overlap-save block rule against resample.ml:279-300 as oracle/ref_ols.py
    restates it; needs no compiled reference, unlike the shaping test below."""
    from oracle import ref_ols
    cfg = lib.Resample.Config.create(sample_rate=sr, target=target)
    rate = sr
    seen = 0
    for s in cfg.stages():
        if s["exec"] == "ols":
            geom = ref_ols.ols_geom(rate, s["l"], s["m"], s["k"])
            assert geom == (s["ols_n"], s["ols_b"], s["ols_delta"]), (sr, target, geom, s)
            seen += 1
        rate = rate * s["l"] // s["m"]
    assert seen >= 1, cfg.pp()


# resample_stubs.c:329-408 (soundml_resample_shape, compiled unmodified into oracle/_ref) inside
# the reference's overlap-save orchestration (oracle/ref_ols.py restates resample.ml:279-300,
# 856-867, 1313-1315, 1456-1598): the reference's OLS surface must equal the oracle's stage
# filter -- which is what every GPU overlap-save kernel is tested against.
@needs_ref
@pytest.mark.parametrize("sr,target", OLS_PAIRS)
def test_reference_ols_shaping_matches_the_oracle_stage_filter(lib, sr, target):
    from oracle import ref_ols
    cfg = lib.Resample.Config.create(sample_rate=sr, target=target)
    rate = sr
    seen = 0
    for s, st in zip(cfg.stages(), oracle_stages(cfg)):
        if s["exec"] == "ols":
            # the planner's block rule is the reference's (plan strings carry N; here also B, delta)
            geom = ref_ols.ols_geom(rate, s["l"], s["m"], s["k"])
            assert geom == (s["ols_n"], s["ols_b"], s["ols_delta"]), (sr, target, geom, s)
            rng = np.random.default_rng(sr + target + s["k"])
            for n in (1, 333, 5 * s["ols_n"] + 17):
                x = rng.uniform(-1, 1, n)
                n_out = R.ceil_div(n * s["l"], s["m"])
                want = R.stage_apply(x[None], st["proto"], s["l"], s["m"], s["k"], n_out)[0]
                got = ref_ols.stage_apply(x, st["proto"], s["l"], s["m"], s["k"], n_out, geom)
                peak = max(np.abs(want).max(), 1e-300)
                assert np.abs(got - want).max() / peak <= 1e-12, (sr, target, n)
            seen += 1
        rate = rate * s["l"] // s["m"]
    assert seen >= 1, cfg.pp()
