"""SqueezeSegV2 model builder - mirrors pcl_segmentation/nets/SqueezeSegV2.py (CAM :30-82, FIRE :85-140,
FIREUP :143-213, SqueezeSegV2 :216-334).  ``call`` is traced symbolically (nets/layers.py) into fused libpclseg ops;
variable names are the Keras attribute paths (conv1/kernel, fire2/squeeze_bn/gamma, ...)."""
from . import layers as L
from .SegmentationNetwork import PCLSegmentationNetwork


class CAM(L.Layer):
  """Context Aggregation Module: x * sigmoid(BN(1x1(relu(BN(1x1(maxpool7x7(x))))))) - ONE fused kernel (cam2_kernel)."""

  def __init__(self, path, in_channels, reduction_factor=16):
    super().__init__(path)
    self.in_channels = in_channels
    self.reduction_factor = reduction_factor

  def __call__(self, inputs, training=False):
    return inputs.graph.cam(inputs, self.path, self.in_channels // self.reduction_factor)


class FIRE(L.Layer):
  """FIRE MODULE"""

  def __init__(self, path, sq1x1_planes, ex1x1_planes, ex3x3_planes):
    super().__init__(path)
    self.squeeze = L.Conv2D(path + "/squeeze", sq1x1_planes, 1)
    self.squeeze_bn = L.BatchNormalization(path + "/squeeze_bn")
    self.expand1x1 = L.Conv2D(path + "/expand1x1", ex1x1_planes, 1)
    self.expand1x1_bn = L.BatchNormalization(path + "/expand1x1_bn")
    self.expand3x3 = L.Conv2D(path + "/expand3x3", ex3x3_planes, 3)
    self.expand3x3_bn = L.BatchNormalization(path + "/expand3x3_bn")

  def __call__(self, inputs, training=False):
    squeeze = L.relu(self.squeeze_bn(self.squeeze(inputs), training))
    expand1x1 = L.relu(self.expand1x1_bn(self.expand1x1(squeeze), training))
    expand3x3 = L.relu(self.expand3x3_bn(self.expand3x3(squeeze), training))
    return L.concat([expand1x1, expand3x3], axis=3)


class FIREUP(L.Layer):
  """FIRE MODULE WITH TRANSPOSE CONVOLUTION (the upconv has a bias and a ReLU but no BatchNorm)"""

  def __init__(self, path, sq1x1_planes, ex1x1_planes, ex3x3_planes, stride):
    super().__init__(path)
    self.stride = stride
    self.squeeze = L.Conv2D(path + "/squeeze", sq1x1_planes, 1)
    self.squeeze_bn = L.BatchNormalization(path + "/squeeze_bn")
    if self.stride == 2:
      self.upconv = L.Conv2DTranspose(path + "/upconv", sq1x1_planes, kernel_size=[1, 4], strides=[1, 2])
    self.expand1x1 = L.Conv2D(path + "/expand1x1", ex1x1_planes, 1)
    self.expand1x1_bn = L.BatchNormalization(path + "/expand1x1_bn")
    self.expand3x3 = L.Conv2D(path + "/expand3x3", ex3x3_planes, 3)
    self.expand3x3_bn = L.BatchNormalization(path + "/expand3x3_bn")

  def __call__(self, inputs, training=False):
    squeeze = L.relu(self.squeeze_bn(self.squeeze(inputs), training))
    if self.stride == 2:
      upconv = L.relu(self.upconv(squeeze))
    else:
      upconv = squeeze
    expand1x1 = L.relu(self.expand1x1_bn(self.expand1x1(upconv), training))
    expand3x3 = L.relu(self.expand3x3_bn(self.expand3x3(upconv), training))
    return L.concat([expand1x1, expand3x3], axis=3)


class SqueezeSegV2(PCLSegmentationNetwork):
  """SqueezeSegV2 Model"""

  def __init__(self, mc):
    super(SqueezeSegV2, self).__init__(mc)
    self.drop_rate = mc.DROP_RATE

    # Encoder
    self.conv1 = L.Conv2D("conv1", 64, 3, strides=[1, 2])
    self.bn1 = L.BatchNormalization("bn1")
    self.cam1 = CAM("cam1", in_channels=64)
    self.conv1_skip = L.Conv2D("conv1_skip", 64, 1)
    self.bn1_skip = L.BatchNormalization("bn1_skip")

    self.fire2 = FIRE("fire2", 16, 64, 64)
    self.cam2 = CAM("cam2", in_channels=128)
    self.fire3 = FIRE("fire3", 16, 64, 64)
    self.cam3 = CAM("cam3", in_channels=128)
    self.fire4 = FIRE("fire4", 32, 128, 128)
    self.fire5 = FIRE("fire5", 32, 128, 128)
    self.fire6 = FIRE("fire6", 48, 192, 192)
    self.fire7 = FIRE("fire7", 48, 192, 192)
    self.fire8 = FIRE("fire8", 64, 256, 256)
    self.fire9 = FIRE("fire9", 64, 256, 256)

    # Decoder
    self.fire10 = FIREUP("fire10", 64, 128, 128, stride=2)
    self.fire11 = FIREUP("fire11", 32, 64, 64, stride=2)
    self.fire12 = FIREUP("fire12", 16, 32, 32, stride=2)
    self.fire13 = FIREUP("fire13", 16, 32, 32, stride=2)

    self.conv14 = L.Conv2D("conv14", self.NUM_CLASS, 3)
    self.dropout = L.Dropout(self.drop_rate)

    self._trace()

  def call(self, inputs, training=False, mask=None):
    lidar_input, lidar_mask = inputs[0], inputs[1]

    # Encoder
    x = self._tap("conv1", L.relu(self.bn1(self.conv1(lidar_input))))
    cam1_output = self._tap("cam1", self.cam1(x))
    conv1_skip = self._tap("conv1_skip", self.bn1_skip(self.conv1_skip(lidar_input)))

    x = L.max_pool2d(cam1_output, ksize=3, strides=[1, 2], padding='SAME')
    x = self._tap("fire2", self.fire2(x))
    x = self.cam2(x)
    x = self.fire3(x)
    cam3_output = self._tap("cam3", self.cam3(x))

    x = L.max_pool2d(cam3_output, ksize=3, strides=[1, 2], padding='SAME')
    x = self.fire4(x)
    fire5_output = self._tap("fire5", self.fire5(x))

    x = L.max_pool2d(fire5_output, ksize=3, strides=[1, 2], padding='SAME')
    x = self.fire6(x)
    x = self.fire7(x)
    x = self.fire8(x)
    fire9_output = self._tap("fire9", self.fire9(x))

    # Decoder (each tf.add skip is folded into the FireDeconv's expand epilogues)
    x = self.fire10(fire9_output)
    x = self._tap("fire10", L.add(x, fire5_output))
    x = self.fire11(x)
    x = L.add(x, cam3_output)
    x = self.fire12(x)
    x = L.add(x, cam1_output)
    x = self.fire13(x)
    x = self._tap("fire13", L.add(x, conv1_skip))

    x = self.dropout(x, training)
    logits = self.conv14(x)
    return self.segmentation_head(logits, lidar_mask)
