"""Host logic of gym_roboy_b200.evaluation (no GPU): the default step count of evaluate_policy."""
from gym_roboy_b200.evaluation import default_n_steps


def test_default_n_steps_follows_the_step_counter_rule():
    """A step counter starts at 1 on reset and an episode ends at the latest when it passes max_episode_len, so an
    episode lasts at most max(max_episode_len, 1) steps: K of them after a reset, one more for the uncounted episode in
    progress without a reset."""
    assert default_n_steps(400, 3) == 1200 and default_n_steps(400, 3, reset=False) == 1600
    assert default_n_steps(400, 1) == 400 and default_n_steps(400, 0) == 0 and default_n_steps(400, 0, reset=False) == 400
    assert default_n_steps(1, 5) == 5 and default_n_steps(0, 2) == 2 and default_n_steps(-3, 2, reset=False) == 3
