"""CPU guard over the shape sweep of tests/test_gpu_shapes.py: the case table reaches every kernel branch the sweep is
meant to cover.  The predicates are restated in test_gpu_shapes.tc_plan / f32_rows / tc_tiles (each commented with the
rollout_tc.cu / rollout_f32.cu line it mirrors; test_plan_restatement_matches_library checks them against the library on
the GPU).  Trimming a case that was the only one to reach a branch fails here instead of quietly losing the branch."""
from test_gpu_shapes import ALL_CASES, B200_SMS, MULTI_TILE, REJECTED, SWEEP, f32_rows, mode_spec, tc_plan, tc_tiles


def _tc_runs():
    """(name, mode, spec, plan) of every tensor-core run of the sweep and the multi-tile cases."""
    out = []
    for name, (spec, modes) in ALL_CASES.items():
        for mode in modes:
            s = mode_spec(spec, mode)
            plan = tc_plan(s, expectation=mode == "expect")
            if plan is not None:
                out.append((name, mode, s, plan))
    return out


def test_hidden_width_residues_and_limits():
    tc = _tc_runs()
    assert {s.hid_size % 16 for _, _, s, _ in tc} == set(range(16))  # the tail chunk's bias columns at every offset
    widths = {s.hid_size for _, _, s, _ in tc}
    assert 17 in widths and 254 in widths  # smallest / largest accepted
    for name, w in (("h16", 16), ("h255", 255)):
        assert REJECTED[name].hid_size == w and tc_plan(REJECTED[name]) is None
    # hid % 16 == 14: bias ones fill the padding exactly; == 15: they straddle Np into the extra K step
    assert any(s.hid_size % 16 == 14 for _, _, s, _ in tc) and any(s.hid_size % 16 == 15 for _, _, s, _ in tc)


def test_depth_activation_and_options():
    tc = _tc_runs()
    assert {s.num_layers for _, _, s, _ in tc} == set(range(1, 8))
    assert {s.activation for _, _, s, _ in tc if s.num_layers >= 4} == {"relu", "silu", "leaky_relu"}
    specs = [s for _, _, s, _ in tc]
    assert any(s.deterministic for s in specs)
    assert any(not s.target_is_delta for s in specs)
    assert any(s.no_delta_list for s in specs)
    assert {s.normalize for s in specs} == {None, "float32", "float64"}
    assert {s.obs_process for s in specs} == {None, "halfcheetah", "cartpole"}
    assert {s.out_size % 4 for s in specs} == {0, 1, 2, 3}
    assert any(s.act_dim <= 8 for s in specs) and any(s.act_dim > 8 for s in specs)
    # L >= 5 with a termination function (judged by the discrete bars)
    assert any(s.num_layers >= 5 and s.term_fn != "no_termination" for s in specs)
    for modes in ("ts1", "tsinf", "shuffle", "expect"):
        assert any(m == modes for _, m, _, _ in tc)


def test_input_and_output_widths():
    tc = _tc_runs()
    ins = {s.in_size + 2 for _, _, s, _ in tc}
    assert any(x % 16 == 15 for x in ins) and any(x % 16 == 1 for x in ins)  # in + 2 just below / above a multiple of 16
    assert any(p["Kp0"] == 256 and s.in_size == 254 for _, _, s, p in tc)   # widest input: Kp0 = 256
    assert any(s.out_size == 128 and 2 * s.out_size == 256 for _, _, s, _ in tc if not s.deterministic)  # nout = 256
    # hid % 16 == 8 below the layer-0 operand width: the generic tail (rollout_tc.cu:523 fails on hid >= Kp0)
    assert any(s.hid_size % 16 == 8 and s.hid_size < p["Kp0"] for _, _, s, p in tc)
    assert any(p["nstages"] == 1 for _, _, _, p in tc)  # one weight-ring stage: no prefetch of the next layer


def test_every_branch_takes_both_values():
    tc = _tc_runs()
    for key in ("fast_tail", "final_early", "fuse_in", "act_regs"):
        assert {p[key] for _, _, _, p in tc} == {True, False}, key
    # the fused next-step input with each activation
    assert {s.activation for _, _, s, p in tc if p["fuse_in"]} == {"relu", "silu", "leaky_relu"}


def test_fp32_row_tiles():
    """rollout_f32.cu:318-332 at 232 448 B of shared memory: every case the sweep runs gets a tile, and the sweep runs
    the 64- and the 32-row instantiation (the 16-row one is Humanoid-v4's, tests/test_gpu_parity.py)."""
    rows = {name: f32_rows(spec) for name, (spec, _) in ALL_CASES.items()}
    assert None not in rows.values()
    assert set(rows.values()) == {64, 32}
    assert rows["h512_f32"] == 32 and tc_plan(SWEEP["h512_f32"][0]) is None


def test_multi_tile_grids():
    sizes = {}
    for name, (spec, modes) in MULTI_TILE.items():
        for mode in modes:
            s = mode_spec(spec, mode)
            assert tc_plan(s, expectation=mode == "expect") is not None, name
            tiles = tc_tiles(s, mode)
            sizes[(name, mode)] = tiles
            if mode == "expect":
                assert tiles > B200_SMS
                assert (s.population * s.particles) % 128 != 0  # partial last tile
            else:
                assert tiles > 2 * B200_SMS, (name, mode, tiles)
                rows = s.population if mode == "shuffle" else s.population * s.particles // s.num_models
                assert rows % 128 != 0  # partial last tile
    cfg2 = MULTI_TILE["config2_H7"][0]
    assert (cfg2.num_layers + 1) * cfg2.horizon % 2 == 1  # a CTA's second tile starts on the other activation buffer
    assert (cfg2.hid_size, cfg2.num_layers, cfg2.num_models) == (200, 4, 5)
    h72 = MULTI_TILE["h72_L5"][0]
    assert h72.hid_size % 16 == 8 and h72.num_layers == 5 and tc_plan(h72)["fast_tail"]  # tail constants once per CTA
    assert {m for _, ms in MULTI_TILE.values() for m in ms} == {"tsinf", "shuffle", "expect"}
