"""Options of the ResNet-50 engine that select a removed variant fail loudly instead of running the default path."""
import pytest

from b200ddl.models.resnet_engine import ResNet50Engine


@pytest.mark.parametrize("option", ["fuse_bn_coeffs", "fuse_stem_bwd"])
def test_removed_variants_raise(option):
    with pytest.raises(ValueError, match="profiles/README.md"):
        ResNet50Engine(batch=8, **{option: True})
