"""B200-native batched discrete-event simulator for LibraBFTv2 (drop-in for the reference's
``bft_lib::simulator`` hot path).  See DESIGN.md and include/lbft.h."""
from .simulator import (BatchResult, BatchSimulator, Command, GlobalTime, NodeConfig, ParamSet, RandomDelay,  # noqa: F401
                        SimulatedContextView, Simulator, format_round_switches_csv, write_data_files)

from .distributed import ShardedBatchSimulator, ShardedResult, shard_bounds  # noqa: F401,E402

__all__ = ["ShardedBatchSimulator", "ShardedResult", "shard_bounds", "BatchResult", "BatchSimulator", "Command", "GlobalTime", "NodeConfig", "ParamSet", "RandomDelay",
           "SimulatedContextView", "Simulator", "format_round_switches_csv", "write_data_files"]
