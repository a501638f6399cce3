"""InformationGainPerUnitCost (robo/acquisition_functions/information_gain_per_unit_cost.py): the information gain of
a configuration divided by its predicted cost plus an optimisation overhead (Swersky et al., NIPS 2013), the
acquisition of the Fabolas facade.  The information gain is InformationGain's device path."""
import numpy as np

from robo_b200.acquisition_functions.information_gain import InformationGain


class InformationGainPerUnitCost(InformationGain):

    def __init__(self, model, cost_model, lower, upper, is_env_variable, sampling_acquisition=None, n_representer=50):
        self.cost_model = cost_model
        self.n_dims = lower.shape[0]
        self.is_env = is_env_variable
        super(InformationGainPerUnitCost, self).__init__(model, lower, upper, sampling_acquisition=sampling_acquisition,
                                                         Nb=n_representer)

    def update(self, model, cost_model, overhead=None):
        self.cost_model = cost_model
        self.overhead = 0 if overhead is None else overhead
        super(InformationGainPerUnitCost, self).update(model)

    def compute(self, X, derivative=False):
        """dh / (exp(log cost) + overhead) (information_gain_per_unit_cost.py:67-106)."""
        if len(X.shape) == 1:
            X = X[np.newaxis, :]
        if derivative:
            raise NotImplementedError("InformationGainPerUnitCost: derivative=True is not supported")
        log_cost = self.cost_model.predict(X)[0]
        dh = super(InformationGainPerUnitCost, self).compute(X, derivative=derivative)
        return dh / (np.exp(log_cost) + self.overhead)

    def argmax(self, X):
        return int(np.argmax(self.compute(X)))

    # representer points live in the configuration space; the environment columns are fixed (:108-154)
    def _sampling_lower_upper(self):
        return self.lower[np.where(self.is_env == 0)], self.upper[np.where(self.is_env == 0)]

    def _project(self, X):
        env = np.broadcast_to(self.upper[self.is_env == 1], (X.shape[0], int(np.sum(self.is_env == 1))))
        return np.concatenate((X, env), axis=1)

    def sampling_acquisition_wrapper(self, x):
        lower, upper = self._sampling_lower_upper()
        if np.any(x < lower) or np.any(x > upper):
            return -np.inf
        return self.sampling_acquisition(self._project(np.array([x])))[0]

    def sample_representer_points(self):
        super(InformationGainPerUnitCost, self).sample_representer_points()
        if np.any(np.isinf(self.lmb)):
            raise ValueError("Could not sample valid representer points! LogEI is -infinity")
        # the environment columns get the NUMBER of environment columns, not upper (the reference's projection, :150-154)
        n_env = self.upper[self.is_env == 1].shape[0]
        self.zb = np.concatenate((self.zb, np.ones([self.zb.shape[0], n_env]) * n_env), axis=1)
