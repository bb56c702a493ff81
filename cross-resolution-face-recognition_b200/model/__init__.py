from .FSRnet import (OverallNetwork, Course_SR_Network, Fine_SR_Encoder, Prior_Estimation_Network, Fine_SR_Decoder,
                     weights_init)  # noqa: F401
from .resnet import ResNet, BasicBlock, ResNet_34  # noqa: F401
from .model_irse import Backbone, IR_50, IR_101, IR_152, IR_SE_50, IR_SE_101, IR_SE_152  # noqa: F401
