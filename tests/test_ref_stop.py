"""Parity pin for rows a9-a12: the reference's OWN stop predictor against the restatement.

oracle/_ref is /root/reference/gp_predictor/src/gp_predictor.cpp compiled UNMODIFIED (stand-in ROS / Eigen headers,
oracle/ref_stubs/; recipe oracle/ref_gp_predictor.py).  Here:
  * oracle/stop_oracle.c (libm trigonometry, trig_mode = 0) must give the same decisions as the reference code and the
    same xy-error trace / final covariance / gain / R_IP to 1e-12 relative (only the rounding inside a matrix product
    may differ: fma chains vs multiply-add),
  * the committed vectors tests/golden/stop_ref_golden.npz (outputs of oracle/_ref, made by
    tests/golden/make_stop_ref_golden.py) must be reproduced by the restatement - this part runs without _ref,
  * the deterministic trigonometry (trig_mode = 1, what the CUDA kernel repeats bit for bit) stays within 1 ulp of libm
    and changes no decision of the fixture.
"""
import os

import numpy as np
import pytest

from corenav_gp_b200 import synthetic as syn
from oracle import ref_gp_predictor as rg
from oracle import stop_oracle as so

GOLD = os.path.join(os.path.dirname(__file__), "golden", "stop_ref_golden.npz")
needs_ref = pytest.mark.skipif(not rg.available(), reason="needs a built oracle/_ref or the reference's source tree "
                                                          "under CNGP_REFERENCE_ROOT")


def rel(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def test_ref_is_built_where_the_reference_source_exists():
    if os.path.exists(os.path.join(rg.REF_ROOT, "gp_predictor", "src", "gp_predictor.cpp")):
        assert rg.build() is not None and os.path.exists(rg.build())
        # the reference source is read in place, never copied into the repo
        repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        assert not os.path.exists(os.path.join(repo, "oracle", "gp_predictor.cpp"))


@needs_ref
@pytest.mark.parametrize("s,seed", [(0.2, 0), (0.45, 1), (0.6, 2), (0.69, 3)])
def test_restatement_equals_reference_code(s, seed):
    rng = np.random.default_rng(seed)
    M = 300
    k = np.arange(M)
    mean = 0.06 * np.exp(-k / 60.0) * rng.uniform(-1, 1) + 0.01 * rng.standard_normal(M)
    sigma = 2.0 * np.sqrt(1e-3 + 0.01 * (1 - np.exp(-k / 150.0))) * rng.uniform(0.7, 1.3)
    if seed == 2:
        mean += 0.4            # large slip: the UT covariance beats the floors (gp_predictor.cpp:80-83)
        sigma *= 2.0
    c = syn.lookahead_context(s)
    r = rg.gp_callback(mean, sigma, c["P"], c["Q"], c["STM"], c["Hvec"], c["pos"])
    o = so.lookahead(mean, sigma, c["P"], c["Q"], c["STM"], c["Hvec"], c["pos"], want_trace=True)
    assert r["triggered"] == o["triggered"]
    assert r["i_stop"] == o["i_stop"] and r["step_stop"] == o["step_stop"]
    n = r["n_steps"]
    assert n == (o["step_stop"] + 1 if o["triggered"] else 5 * M)
    assert np.max(np.abs(r["xy_trace"] - o["xy_trace"][:n]) / np.abs(r["xy_trace"])) < 1e-12
    assert abs(r["xy_err"] - o["xy_err"]) < 1e-12 * r["xy_err"]
    assert rel(o["P"], r["P"]) < 1e-12
    # the reference leaves R_IP / K_pred at their last update (public members, gp_predictor.h:36-39)
    assert rel(so.ut_R(mean[r["i_stop"] - 1], sigma[r["i_stop"] - 1]), r["R"]) < 1e-14


@needs_ref
def test_published_stop_time_follows_the_reference_clock_rule():
    """gp_predictor.cpp:107-116: stop_cmd = gp_arrived + i/10 - now, or 0.5 when that is negative."""
    c = syn.lookahead_context(0.5)
    M = 200
    mean, sigma = np.full(M, 0.05), np.full(M, 0.2)
    r0 = rg.gp_callback(mean, sigma, c["P"], c["Q"], c["STM"], c["Hvec"], c["pos"])
    assert r0["triggered"] and r0["stop_cmd"] == r0["i_stop"] / 10.0
    late = rg.gp_callback(mean, sigma, c["P"], c["Q"], c["STM"], c["Hvec"], c["pos"], clock_arrive=100.0,
                          clock_later=100.0 + r0["i_stop"] / 10.0 + 1.0)
    assert late["stop_cmd"] == 0.5
    early = rg.gp_callback(mean, sigma, c["P"], c["Q"], c["STM"], c["Hvec"], c["pos"], clock_arrive=100.0,
                           clock_later=100.25)
    assert early["stop_cmd"] == 100.0 + r0["i_stop"] / 10.0 - 100.25


@needs_ref
def test_h_aliasing_is_the_reference_behaviour():
    """The reference reads HvecData[r*4+c] (gp_predictor.cpp:38-42): the restatement with fix_h_packing = 0 equals it,
    and the 'intended' packing does not."""
    c = syn.lookahead_context(0.45)
    M = 120
    mean, sigma = np.full(M, 0.03), np.full(M, 0.15)
    r = rg.gp_callback(mean, sigma, c["P"], c["Q"], c["STM"], c["Hvec"], c["pos"])
    o = so.lookahead(mean, sigma, c["P"], c["Q"], c["STM"], c["Hvec"], c["pos"], want_trace=True)
    assert np.max(np.abs(r["xy_trace"] - o["xy_trace"][:r["n_steps"]]) / np.abs(r["xy_trace"])) < 1e-12
    hv = c["H"].reshape(60)
    o_fix = so.lookahead(mean, sigma, c["P"], c["Q"], c["STM"], hv, c["pos"], so.default_cfg(fix_h_packing=1),
                         want_trace=True)
    n = min(r["n_steps"], o_fix["step_stop"] + 1)
    assert np.max(np.abs(r["xy_trace"][:n] - o_fix["xy_trace"][:n]) / np.abs(r["xy_trace"][:n])) > 1e-6


@needs_ref
def test_llh_to_enu_equals_reference_code():
    rng = np.random.default_rng(4)
    for p in syn.INIT_LLH[None, :] + rng.normal(0, [1e-4, 1e-4, 20.0], (32, 3)):
        a, b = rg.llh_to_enu(*p), so.llh_to_enu(*p)
        assert np.max(np.abs(a - b)) < 2e-9       # metres: ulp(6.4e6) = 9e-10; products R*d are fma vs mul+add


@needs_ref
def test_golden_file_is_what_the_reference_code_returns():
    g = np.load(GOLD)
    for b in (0, 1, 2, 17, 35, 47):
        r = rg.gp_callback(g["mean"][b], g["sigma"][b], g["P"][b], g["Q"][b], g["STM"][b], g["Hvec"][b], g["pos"][b])
        assert r["triggered"] == bool(g["triggered"][b]) and r["i_stop"] == g["i_stop"][b]
        assert r["xy_err"] == g["xy_err"][b] and np.array_equal(r["P"].ravel(), g["P_final"][b])


@pytest.mark.parametrize("trig_mode", [0, 1])
def test_restatement_reproduces_the_golden_vectors(trig_mode):
    """Runs anywhere (no _ref needed): reference outputs committed as a fixture."""
    g = np.load(GOLD)
    B = g["mean"].shape[0]
    cfg = so.default_cfg(trig_mode=trig_mode)
    out = so.lookahead_batch(g["mean"], g["sigma"], g["P"], g["Q"], g["STM"], g["Hvec"], g["pos"], cfg)
    assert 0 < g["triggered"].sum() < B
    assert np.array_equal(out["triggered"], g["triggered"])
    assert np.array_equal(out["i_stop"], g["i_stop"])
    assert np.array_equal(out["step_stop"], g["step_stop"])
    tol = 1e-12 if trig_mode == 0 else 1e-9      # 1 ulp of sin/cos on ECEF-sized intermediates is ~1e-9 m
    assert np.max(np.abs(out["xy_err"] - g["xy_err"]) / g["xy_err"]) < tol
    b = int(g["trace0_window"])
    o = so.lookahead(g["mean"][b], g["sigma"][b], g["P"][b], g["Q"][b], g["STM"][b], g["Hvec"][b], g["pos"][b], cfg,
                     want_trace=True)
    n = g["trace0"].size
    assert np.max(np.abs(o["xy_trace"][:n] - g["trace0"]) / g["trace0"]) < tol
    assert rel(o["P"].ravel(), g["P_final"][b]) < 1e-12
    enu = np.stack([so.llh_to_enu(*p, cfg) for p in g["enu_in"]])
    assert np.max(np.abs(enu - g["enu_out"])) < (2e-9 if trig_mode == 0 else 5e-9)


def test_restatement_reproduces_the_golden_state_and_stop_time():
    """Runs anywhere: for every window of the fixture (a fifth of them with large slip, where the UT covariance beats the
    floors of gp_predictor.cpp:80-83), P_pred / K_pred / R_IP as the reference leaves them in its public members
    (gp_predictor.h:36-43), and the stop time it published under a constant clock (gp_predictor.cpp:107-116: i/10;
    nothing without a trigger)."""
    g = np.load(GOLD)
    for b in range(g["mean"].shape[0]):
        mean, sigma = g["mean"][b], g["sigma"][b]
        o = so.lookahead(mean, sigma, g["P"][b], g["Q"][b], g["STM"][b], g["Hvec"][b], g["pos"][b])
        assert rel(o["P"].ravel(), g["P_final"][b]) < 1e-12
        assert rel(o["K"].ravel(), g["K_final"][b]) < 1e-11
        assert rel(o["R"].ravel(), g["R_final"][b]) < 1e-14
        assert rel(so.ut_R(mean[o["i_stop"] - 1], sigma[o["i_stop"] - 1]).ravel(), g["R_final"][b]) < 1e-14
        if o["triggered"]:
            assert o["i_stop"] / 10.0 == g["stop_cmd"][b]
        else:
            assert np.isnan(g["stop_cmd"][b])


def test_golden_trace_follows_the_aliased_h_packing():
    """Runs anywhere: the reference reads HvecData[r*4+c] (gp_predictor.cpp:38-42).  The fixture's Hvec is that packing
    of the synthetic H, its stored trace is reproduced with fix_h_packing = 0 (test above), and the 'intended' packing
    departs from it."""
    g = np.load(GOLD)
    b = int(g["trace0_window"])
    H = syn.lookahead_context(0.5)["H"]
    assert np.array_equal(syn.pack_hvec(H), g["Hvec"][b])
    o_fix = so.lookahead(g["mean"][b], g["sigma"][b], g["P"][b], g["Q"][b], g["STM"][b], H.reshape(60), g["pos"][b],
                         so.default_cfg(fix_h_packing=1), want_trace=True)
    n = min(g["trace0"].size, o_fix["step_stop"] + 1)
    assert np.max(np.abs(g["trace0"][:n] - o_fix["xy_trace"][:n]) / np.abs(g["trace0"][:n])) > 1e-6


def test_deterministic_trig_is_within_one_ulp_of_libm():
    rng = np.random.default_rng(7)
    xs = np.concatenate([rng.uniform(-4, 4, 20000), rng.uniform(-1e5, 1e5, 2000),
                         [0.0, np.pi / 2, np.pi, -np.pi / 4, syn.INIT_LLH[0], syn.INIT_LLH[1], 1e-300]])
    worst = 0.0
    for x in xs:
        s, c = so.det_sincos(x)
        worst = max(worst, abs(s - np.sin(x)) / np.spacing(abs(np.sin(x))), abs(c - np.cos(x)) / np.spacing(abs(np.cos(x))))
    assert worst <= 1.0, worst
