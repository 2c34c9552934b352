from .fpn_fabu import fpn_r50_fabu, SemanticFPNFabu  # noqa: F401
