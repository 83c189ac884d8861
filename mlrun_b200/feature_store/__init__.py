from . import steps  # noqa: F401
from .infer import InferOptions  # noqa: F401
