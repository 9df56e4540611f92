"""GPU parity of the ground-truth simulator (cbo_sem_eval, csrc/sem.cu) against the host function it replaces --
compute_interventions, reference graph_functions.py:48-77 (100 000 SEM samples per intervention, reseeded with seed 1 on
every call) -- and against the true causal effects shipped with the reference (data/*/interventional_data.npy)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = [("toy_graph", ["X"]), ("toy_graph", ["Z"]), ("complete_graph", ["B"]), ("complete_graph", ["D", "E"]),
         ("complete_graph", ["B", "E"]), ("coral_graph", ["N"]), ("coral_graph", ["O", "T"]), ("coral_graph", ["N", "C", "D"]),
         ("simplified_coral_graph", ["O", "C", "T"])]


@pytest.mark.parametrize("experiment,variables", CASES, ids=lambda v: v if isinstance(v, str) else "".join(v))
def test_device_sem_equals_host_function(cuda_engine_ready, experiment, variables):
    from cbo_with_oop_b200.sem import DeviceSEM
    from src.DataLoader import DataLoader
    from src.utils_functions.graph_functions import compute_interventions
    np.random.seed(3)
    g = DataLoader(experiment, 100).graph
    ranges = g.get_interventional_ranges()
    rng = np.random.default_rng(11)
    X = np.column_stack([rng.uniform(ranges[v][0], ranges[v][1], 5) for v in variables])
    n = 20000
    sim = DeviceSEM(g, num_samples=n)
    state = np.random.get_state()
    got = sim.mean_target(variables, X)                     # one launch for the batch of 5 interventions
    assert all(np.array_equal(a, b) if isinstance(a, np.ndarray) else a == b for a, b in zip(state, np.random.get_state())), \
        "the device path must not disturb the caller's NumPy stream"
    sem = g.define_sem()
    for b in range(len(X)):
        ref = compute_interventions(sem, {v: "" for v in variables}, X[b:b + 1], num_samples=n)[0, 0]
        assert abs(got[b] - ref) <= 1e-12 * max(1.0, abs(ref)), (b, got[b], ref)
    # a second call reuses the resident noise and returns the same bits (deterministic summation order)
    np.testing.assert_array_equal(sim.mean_target(variables, X), got)


def test_device_sem_matches_shipped_true_effects(cuda_engine_ready):
    """E[Y | do(.)] by the device Monte Carlo against the true causal effects the reference ships (statistical tolerance)."""
    from cbo_with_oop_b200.sem import DeviceSEM
    from src.DataLoader import DataLoader
    data = DataLoader("toy_graph", 100)
    sim = DeviceSEM(data.graph, num_samples=200000)
    xz, yz = data.interventions[1][2], data.interventions[1][3]            # row 'Z': x (20, 1), true effect (20, 1)
    got = sim.mean_target(["Z"], xz)
    assert np.abs(got - yz[:, 0]).max() < 0.02
    data = DataLoader("complete_graph", 100)
    sim = DeviceSEM(data.graph, num_samples=200000)
    row = [r for r in data.interventions if [str(v) for v in r[1:1 + int(r[0])]] == ["B", "D"]][0]
    got = sim.mean_target(["B", "D"], np.asarray(row[3], np.float64))
    assert np.abs(got - np.asarray(row[4], np.float64).reshape(-1)).max() < 0.05


def test_monitor_uses_the_device_simulator(cuda_engine_ready, tmp_path, monkeypatch):
    import types
    from src.CBO import CBO
    from src.DataLoader import DataLoader
    from src.utils_functions.graph_functions import compute_interventions
    monkeypatch.chdir(tmp_path)          # the agent creates ./data/<experiment>/... for its results
    args = types.SimpleNamespace(exploration_set="MIS", initial_num_obs_samples=60, num_interventions=10, type_cost=1,
                                 num_additional_observations=20, num_trials=3, name_index=0, seed=9, causal_prior=True,
                                 experiment="complete_graph", task="min", grid_points=20, device="cuda:0", num_sem_samples=5000)
    np.random.seed(9)
    cbo = CBO(args, DataLoader("complete_graph", 60), verbose=False)
    x = np.array([[0.3, -0.7]])
    y_dev = cbo.monitor.target_function_list[3](x)                          # set ['B', 'D']
    y_host = compute_interventions(cbo.graph.define_sem(), {"B": "", "D": ""}, x, num_samples=5000)
    assert y_dev.shape == (1, 1) and abs(y_dev[0, 0] - y_host[0, 0]) <= 1e-12 * max(1.0, abs(y_host[0, 0]))
