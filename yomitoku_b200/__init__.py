"""yomitoku_b200: Blackwell-native DBNet -> PARSeq OCR hot path behind yomitoku's module API.

    from yomitoku_b200 import OCR, TextDetector, TextRecognizer, DocumentAnalyzer
    from yomitoku_b200 import LayoutAnalyzer, LayoutParser, TableStructureRecognizer, CellDetector

The constructors, the `configs` dict and the call contracts mirror kotaro-kinoshita/yomitoku
(src/yomitoku/{text_detector,text_recognizer,ocr,document_analyzer,layout_parser,table_structure_recognizer,
table_cell_detector,layout_analyzer}.py); the models (DBNet++, PARSeq, RT-DETRv2) run as hand-written sm_100a CUDA
kernels behind the C ABI in include/yomitoku_b200.h (libytk_b200.so).
"""
from .document_analyzer import DocumentAnalyzer
from .layout_analyzer import LayoutAnalyzer
from .layout_parser import LayoutParser
from .ocr import OCR
from .table_cell_detector import CellDetector
from .table_structure_recognizer import TableStructureRecognizer
from .text_detector import TextDetector
from .text_recognizer import TextRecognizer

__all__ = ["OCR", "TextDetector", "TextRecognizer", "DocumentAnalyzer", "LayoutAnalyzer", "LayoutParser",
           "TableStructureRecognizer", "CellDetector"]
