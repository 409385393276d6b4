"""``archs.__dict__[config.arch](config)`` registry, as in the reference
(code/archs/__init__.py:1-3; used at code/scripts/cluster/cluster_sobel_twohead.py:174)."""
from .cluster import *
from .segmentation import *
from .semisup import *
