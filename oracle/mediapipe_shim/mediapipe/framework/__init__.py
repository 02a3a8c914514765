from . import formats  # noqa: F401
