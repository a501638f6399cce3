from .bayesian_optimization import bayesian_optimization  # noqa: F401
from .entropy_search import entropy_search  # noqa: F401
