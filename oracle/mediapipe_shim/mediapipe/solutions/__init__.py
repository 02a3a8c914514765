from . import drawing_styles, drawing_utils, face_mesh  # noqa: F401
