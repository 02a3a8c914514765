from . import landmark_pb2  # noqa: F401
