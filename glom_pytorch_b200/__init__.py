"""B200-native GLOM column-update engine behind the glom-pytorch `Glom` API."""
from ._native import GlomB200Error, LIB_PATH
from .contrastive import column_contrastive_loss
from .glom import Glom
from .islands import Islands, islands

__all__ = ["Glom", "GlomB200Error", "LIB_PATH", "Islands", "islands", "column_contrastive_loss"]
