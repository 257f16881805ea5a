# mirrors decoders/__init__.py for the recognition heads and the DB text detector (SegDetector, L1BalanceCELoss)
from .attention_decoder import AttentionDecoder  # noqa: F401
from .ctc_decoder import CTCDecoder  # noqa: F401
from .crnn import CRNNDecoder  # noqa: F401
from .ctc_decoder2d import CTCDecoder2D  # noqa: F401
from .ctc_loss2d import CTCLoss2D, CTC2DLoss  # noqa: F401
from .east import EASTDecoder  # noqa: F401
from .seg_detector import SegDetector  # noqa: F401
from .seg_detector_loss import SegDetectorLossBuilder, L1BalanceCELoss  # noqa: F401
