from .synthetic import SyntheticEnv, SyntheticPixelEnv, SyntheticMixedEnv  # noqa: F401
from .exp_sender_wrapper import (ExpSenderWrapperMultiStepMovingWindowWithInfo,  # noqa: F401
                                 ExpSenderWrapperSSARNStepBootstrap)
