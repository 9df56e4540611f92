"""Causal Bayesian Optimisation agent (reference: src/CBO.py) with the acquisition sweep on the GPU.

Same constructor, attributes and methods as the reference (`run`, `observe`, `intervene`, `epsilon`,
`update_all_gaussian_processes`, `update_gaussian_process_of_last_intervention`, `compute_best_acquisition_values`,
`select_next_intervention`, `compute_cost`, ...).  `compute_best_acquisition_values` is the batched override the
survey asks for: every exploration set's candidates go through one AcquisitionSession pass
(cbo_with_oop_b200: exp tables -> prior precompute -> prior -> batched posterior fit -> EI / cost -> argmax) and the
method still returns `xs, ys` with the reference's shapes, so selection, cost and the Monitor work unchanged."""
from pathlib import Path

import numpy as np
import pandas as pd
from numpy.random import uniform

from src.DoCalculus import DoCalculus
from src.GaussianProcessFactory import GaussianProcessFactory as GPFactory
from src.GaussianProcessFactory import GaussianProcessType as GPType
from src.Monitor import Monitor
from src.utils_functions import *  # noqa: F401,F403


class CBO:
    def __init__(self, args, data, verbose=True):
        self.graph = data.graph
        self.measurements = data.measurements
        self.all_measurements = data.all_measurements
        self.interventions = data.interventions

        self.exploration_set = self.graph.get_exploration_set(args.exploration_set)
        self.es_size = len(self.exploration_set)
        self.num_interventions = args.num_interventions
        self.max_n = args.initial_num_obs_samples + 50
        self.initial_num_obs_samples = args.initial_num_obs_samples
        self.gp_type = GPType.CAUSAL_GP if args.causal_prior else GPType.NON_CAUSAL_GP
        self.num_trials = args.num_trials
        self.task = args.task
        self.num_additional_observations = args.num_additional_observations
        self.type_cost = args.type_cost
        self.name_index = args.name_index
        # build-specific knobs (optional attributes of args)
        self.grid_points_per_dim = getattr(args, "grid_points", 100)
        self.device = getattr(args, "device", "cuda:0")
        self.num_sem_samples = getattr(args, "num_sem_samples", 100000)
        # where observe() fits the observational GPs: "device" (cbo_obs_gp_fit / cbo_obs_gp_nll, the default) or, on explicit
        # request only, "host" (SciPy; input preparation for machines without a GPU -- the sweep itself has no CPU path)
        self.observational_fit = getattr(args, "observational_fit", "device")
        # refine each set's grid maximum off the grid (SweepEngine.refine): the reference's continuous L-BFGS polish
        self.refine_acquisition = bool(getattr(args, "refine_acquisition", False))
        # fit each set's GP variance / lengthscale by marginal likelihood at every refit (K8); off: the reference's (1, 1)
        self.optimize_surrogates = bool(getattr(args, "optimize_surrogates", False))

        self.mean_functions, self.var_functions, self.models = [], [], []
        self.costs = self.graph.get_cost_structure(type_cost=self.type_cost)
        self.saving_dir = self.get_saving_dir(args.experiment, args.num_interventions)
        Path(self.saving_dir).mkdir(parents=True, exist_ok=True)
        self.intervention_names = ["".join(variables) for variables in self.exploration_set]
        self.x_mean = {name: {} for name in self.intervention_names}
        self.x_var = {name: {} for name in self.intervention_names}
        self.monitor = Monitor(self, verbose=verbose)
        self.do_calculus = DoCalculus(self)
        self._plain_session = None        # session of the non-causal surrogates
        self.verbose = verbose

    def get_saving_dir(self, experiment, num_interventions):
        cost_types = ["fix_equal", "fix_different", "fix_different_variable", "fix_equal_variable"]
        return f"./data/{experiment}/{cost_types[self.type_cost - 1]}/{self.initial_num_obs_samples}/{num_interventions}/"

    # ---- main loop (reference :83-121) ----------------------------------------------------------------
    def run(self):
        if self.verbose is True:
            print(f"Exploring {self.exploration_set} with CEO and Causal prior = {self.gp_type}")
        self.observe()
        self.intervene()
        self.monitor.start()
        for _ in range(self.num_trials - 2):
            if uniform(0.0, 1.0) < self.epsilon:
                self.observe()
            else:
                self.intervene()
        self.monitor.stop()
        self.monitor.save_results()
        if self.verbose is True:
            print("=================================== Saved results ===================================")
            print("exploration_set: ", self.exploration_set)
            print("causal_prior: ", self.gp_type)
            print("type_cost: ", self.type_cost)
            print("total_time: ", self.monitor.total_time)
            print("folder: ", self.saving_dir)
            print("=====================================================================================")
            print()

    def observe(self):
        """Collect observations, refit the observational GPs, refresh the do-functions (reference :123-141)."""
        self.monitor.log_agent_behaviour(act=False)
        self.measurements = pd.concat([self.measurements, self.get_new_observation()])
        if self.gp_type == GPType.CAUSAL_GP:
            fit_device = self.device if self.observational_fit == "device" else None
            gaussian_processes = self.graph.fit_all_gaussian_processes(self.measurements, device=fit_device)
            self.mean_functions, self.var_functions = self.do_calculus.update_all_do_functions(gaussian_processes)
        else:
            self.mean_functions, self.var_functions = [None] * self.es_size, [None] * self.es_size
        self.monitor.log_agent_performance()

    def intervene(self):
        """One acquisition sweep and the chosen intervention (reference :143-173)."""
        self.monitor.log_agent_behaviour(act=True)
        current_best = self.current_best_solution()
        if self.monitor.agent_previously_observed():
            self.update_all_gaussian_processes()
        else:
            self.update_gaussian_process_of_last_intervention()
        acquisition_xs, acquisition_ys = self.compute_best_acquisition_values(current_best)
        intervention_set, intervention = self.select_next_intervention(acquisition_ys)
        current_cost = self.compute_cost(intervention_set, intervention, acquisition_xs)
        self.monitor.log_agent_performance(intervention_set, intervention, acquisition_xs, current_cost)
        self.models[intervention].optimize()

    @property
    def epsilon(self):
        coverage_total = compute_coverage(self.measurements, self.graph.manipulative_variables, self.interventional_ranges)[2]
        coverage_obs = update_hull(self.measurements, self.graph.manipulative_variables)
        rescale = self.measurements.shape[0] / self.max_n
        return (coverage_obs / coverage_total) / rescale

    @property
    def interventional_ranges(self):
        return self.graph.get_interventional_ranges()

    def get_new_observation(self):
        return observe(num_observation=self.num_additional_observations, complete_dataset=self.all_measurements,
                       initial_num_obs_samples=self.initial_num_obs_samples)

    # ---- surrogates ------------------------------------------------------------------------------------
    def _make_model(self, s):
        model = GPFactory.create(self.gp_type, self.monitor.data_x[s], self.monitor.data_y[s],
                                 [self.mean_functions[s], self.var_functions[s]], emukit_wrapper=True)
        if self.gp_type != GPType.CAUSAL_GP:
            model.attach(self.get_plain_session, s)
        return model

    def update_all_gaussian_processes(self):
        self._plain_session = None
        self.models = [self._make_model(s) for s in range(self.es_size)]

    def update_gaussian_process_of_last_intervention(self):
        last = self.monitor.last_intervention
        self.models[last] = self._make_model(last)

    def get_plain_session(self):
        if self._plain_session is None:
            from cbo_with_oop_b200.engine import SetProblem
            from cbo_with_oop_b200.session import AcquisitionSession
            problems = []
            for s, variables in enumerate(self.exploration_set):
                fix, variable = self.graph.fixed_cost_of(variables, self.type_cost)
                problems.append(SetProblem.non_causal(self.monitor.space_list[s].grid_tables(self.grid_points_per_dim),
                                                      self.monitor.data_x[s], self.monitor.data_y[s].reshape(-1), fix, variable,
                                                      name="".join(variables)))
            self._plain_session = AcquisitionSession(problems, device=self.device, fit_hyperparameters=self.optimize_surrogates)
        return self._plain_session

    def get_session(self):
        return self.do_calculus.get_session() if self.gp_type == GPType.CAUSAL_GP else self.get_plain_session()

    def compute_best_acquisition_values(self, current_best):
        """xs[s] (1, d_s) and ys[s] (1, 1): the maximiser and maximum of EI / cost of every exploration set
        (reference :237-260 loops find_next_y_point over the sets; here all sets share one device pass)."""
        session = self.get_session()
        for s, model in enumerate(self.models):
            session.mark_interventional(s, model.X, model.Y)
        out = session.best_per_set(float(current_best), self.task, refine=self.refine_acquisition)
        if self.refine_acquisition:
            xs = [np.asarray(out.set_x[s], np.float64).reshape(1, -1) for s in range(self.es_size)]
        else:
            xs = [session.grid_point(s, out.set_indices[s]).reshape(1, -1) for s in range(self.es_size)]
        ys = [np.array([[out.set_values[s]]]) for s in range(self.es_size)]
        self.last_sweep = out
        return xs, ys

    def current_best_solution(self):
        return find_current_global(self.monitor.current_best_y, self.intervention_names, self.task)

    def select_next_intervention(self, acquisition_ys):
        """First exploration set attaining the maximum acquisition value (reference :269-277)."""
        values = np.asarray(acquisition_ys, np.float64).reshape(-1)
        values = np.where(np.isnan(values), -np.inf, values)
        index = int(np.where(values == np.max(values))[0][0])
        self.monitor.last_intervention = index
        return self.exploration_set[index], index

    def compute_cost(self, intervention_set, intervention, acquisition_xs):
        x = {var: acquisition_xs[intervention][0, i] for i, var in enumerate(intervention_set)}
        return total_cost(intervention_set, self.costs, x)
