"""Mirror of reference models/arcface_model.py (the symbols on the LFAN path)."""
from ..modules import Backbone, Flatten, SEModule, bottleneck_IR, bottleneck_IR_SE, get_blocks  # noqa: F401
