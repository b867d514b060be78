"""blutils_b200 -- B200-native consensus-identity stage of blutils (`blu blastn build-consensus`).

The package holds only what that one hot path needs: `csrc/` (sm_100a CUDA kernels + the C ABI declared in
include/blu_consensus.h) and the host-side mirror of the reference interface (`consensus.py`)."""
from .consensus import (ConsensusBean, ConsensusEngine, ConsensusOutput, ConsensusPanic, ConsensusStrategy, CudaUnavailable, CustomTaxon,
                        MappedErrors, OutputFormat, ParallelBlastOutput, QueryWithConsensus, QueryWithoutConsensus, Taxon, TaxonomyBean,
                        Unsupported, build_consensus_identities, parse_consensus_as_tabular, run_device_resident_configs, run_file_configs,
                        run_host_configs, shard_cuts, shard_cuts_file, write_blutils_output)

__all__ = [n for n in dir() if not n.startswith("_")]
