"""Semi-supervised heads (code/archs/semisup/__init__.py)."""
from .sup_head5 import *
