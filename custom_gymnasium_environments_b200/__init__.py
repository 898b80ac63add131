"""B200-native batched environment engine for the step()/reset() hot path of
hasnainfarid/Custom_Gymnasium_Environments (snake_env_classic first; crypto_trading_env and
traffic_management_env follow).  Host code is Python/PyTorch over a C-ABI CUDA library
(include/beng.h, csrc/); there is no CPU fallback.
"""
from . import _lib
from ._build import build_library
from .builder import BatchedWorldBuilderEnv, WorldBuilderEnv
from .climate import BatchedSmartClimateEnv, SmartClimateEnv
from .crypto import BatchedCryptoTradingEnv, CryptoTradingEnv, TradingConfig
from .normalize import RunningMeanStd, VecNormalize
from .snake import BatchedSnakeEnv, SnakeEnvClassic
from .traffic import BatchedTrafficManagementEnv, TrafficManagementEnv
from .registration import register_all

__all__ = ["BatchedSnakeEnv", "SnakeEnvClassic", "BatchedCryptoTradingEnv", "CryptoTradingEnv", "TradingConfig", "BatchedSmartClimateEnv", "SmartClimateEnv", "BatchedWorldBuilderEnv", "WorldBuilderEnv", "BatchedTrafficManagementEnv", "TrafficManagementEnv", "VecNormalize", "RunningMeanStd", "build_library", "register_all", "_lib"]
__version__ = "0.1.0"

register_all()
