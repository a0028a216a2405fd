"""jackalope_b200 -- B200-native (CUDA sm_100a) Illumina read generation with
jackalope's ``illumina()`` argument surface.  See DESIGN.md."""
from .genome import Haplotypes, HapChromMuts, RefGenome, create_genome, random_genome, random_haplotypes  # noqa: F401
from .illumina import Context, check_illumina_args, default_context, illumina  # noqa: F401
from .mutate import (HapsInfo, SubModel, Tree, create_haplotypes, haps_phylo, haps_theta, sub_F81, sub_F84,  # noqa: F401
                     sub_GTR, sub_HKY85, sub_JC69, sub_K80, sub_TN93, sub_UNREST)
from .pacbio import check_pacbio_args, pacbio, sample_read_plan  # noqa: F401
from .profiles import (JackalopeError, builtin_illumina_profiles, find_profile_file, flatten_profile,  # noqa: F401
                       format_profile, read_profile, seq_sys_by_read_length)

__all__ = ["illumina", "pacbio", "create_genome", "create_haplotypes", "haps_phylo", "haps_theta", "sub_JC69", "sub_K80",
           "sub_F81", "sub_HKY85", "sub_F84", "sub_TN93", "sub_GTR", "sub_UNREST", "Context", "RefGenome", "Haplotypes", "HapChromMuts", "random_genome", "random_haplotypes",
           "read_profile", "flatten_profile", "JackalopeError"]
