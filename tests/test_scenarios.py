"""Scenario constants and tables vs SURVEY.md Appendix B (reference file:line there)."""
import math
import os

import numpy as np

from rl_collision_avoidance_b200 import _lib
from rl_collision_avoidance_b200.scenarios import COMMON, fill_config, make_scenario


def test_constants_match_reference():
    s1, s2, sc = make_scenario('stage1'), make_scenario('stage2'), make_scenario('circle')
    assert (s1.robots_per_world, s2.robots_per_world, sc.robots_per_world) == (24, 44, 50)
    assert (s1.timeout, s2.timeout, sc.timeout) == (150, 200, 10000)
    assert (s1.w_threshold, s2.w_threshold, sc.w_threshold) == (1.05, 1.05, 0.7)
    assert (s1.pre_distance_zero, s2.pre_distance_zero, sc.pre_distance_zero) == (0, 1, 1)
    assert COMMON['goal_radius'] == 0.5 and COMMON['reward_arrive'] == 15 and COMMON['reward_collision'] == -15
    assert COMMON['progress_gain'] == 2.5 and COMMON['range_max'] == 6.0 and COMMON['dt'] == 0.1
    assert (s1.map.resolution, s2.map.resolution, sc.map.resolution) == (0.2, 0.2, 0.01)
    assert s2.groups == (0, 6, 10, 15, 19, 24, 34, 44)


def test_tables():
    s2 = make_scenario('stage2')
    assert s2.init_tab.shape == (44, 4) and s2.goal_tab.shape == (44, 4)
    assert np.allclose(s2.init_tab[0, :3], [-7.0, 11.5, math.pi])
    assert np.allclose(s2.goal_tab[0, :2], [-18.0, 11.5])
    assert s2.init_tab[:34, 3].sum() == 0 and s2.init_tab[34:, 3].sum() == 10      # stage_world2.py:211
    assert s2.goal_tab[:34, 2].sum() == 0 and s2.goal_tab[34:, 2].sum() == 10      # stage_world2.py:165
    # world-file agent poses equal the init table (worlds/stage2.world:113-165 vs model/utils.py:41-53)
    wf = s2.map.init_poses
    assert np.allclose(np.cos(wf[:, 2]), np.cos(s2.init_tab[:, 2]), atol=1e-6)
    assert np.allclose(wf[:, :2], s2.init_tab[:, :2])
    c = make_scenario('circle')
    k = np.arange(50)
    assert np.allclose(c.init_tab[:, 0], np.round(25 * np.cos(2 * np.pi * k / 50), 2), atol=0.011)
    assert np.allclose(c.goal_tab[:, :2], -c.init_tab[:, :2], atol=1e-6)           # antipodal goals


def test_fill_config_derived_fields():
    cfg = fill_config(_lib.EnvConfig(), make_scenario('stage1'), num_worlds=171, beams=512, seed=5)
    assert cfg.ppm == 5.0 and cfg.range_cells == 30.0 and abs(cfg.inv_dt - 10.0) < 1e-5
    assert cfg.grid_w % 16 == 0 and cfg.raw_beams == 512 and cfg.seed == 5
    assert cfg.robots_per_world * cfg.num_worlds == 4104


def test_assets_reproduce_from_reference_worlds():
    """The packaged maps are what the world loader makes of the reference's own world files and bitmaps, which are
    stored unmodified as fixtures under tests/golden/worlds/."""
    from rl_collision_avoidance_b200.worldfile import load_world
    worlds = os.path.join(os.path.dirname(__file__), 'golden', 'worlds')
    for name in ('stage1', 'stage2'):
        m = load_world(os.path.join(worlds, f'{name}.world'))
        a = make_scenario(name).map
        assert np.array_equal(m.cells, a.cells) and (m.origin_cx, m.origin_cy) == (a.origin_cx, a.origin_cy)
