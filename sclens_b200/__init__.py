"""sclens_b200 - B200-native drop-in for the scLENS.sclens() signal-detection path."""
from .api import Handle, apply_umap, clustering, df2sparr, get_denoised_df, sclens  # noqa: F401
from ._lib import SCL_GRAM_FP16, SCL_GRAM_FP16X3, SclError  # noqa: F401

__all__ = ["sclens", "get_denoised_df", "apply_umap", "clustering", "Handle", "df2sparr", "SclError", "SCL_GRAM_FP16", "SCL_GRAM_FP16X3"]
