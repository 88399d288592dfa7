"""Result types of the hot path (pydantic), mirroring reference src/yomitoku/schemas/document_analyzer.py:137-180,
234-254, schemas/table_semantic_parser.py:62-140 (the cell detector's results) and BaseSchema (base.py:51-57): extra
fields forbidden, assignment validated."""
from typing import Any, Dict, List, Union

from pydantic import BaseModel, ConfigDict, Field, conlist

Quad = conlist(conlist(int, min_length=2, max_length=2), min_length=4, max_length=4)


class BaseSchema(BaseModel):
    model_config = ConfigDict(extra="forbid", validate_assignment=True)

    def to_json(self, out_path: str, **kwargs):
        import json
        with open(out_path, "w", encoding="utf-8") as f:
            json.dump(self.model_dump(), f, ensure_ascii=False, indent=kwargs.get("indent", 4))


class WordPrediction(BaseSchema):
    points: Quad = Field(..., description="[[x1, y1], [x2, y2], [x3, y3], [x4, y4]]")
    content: str = Field(..., description="Text content of the word")
    direction: str = Field(..., description="'horizontal' or 'vertical'")
    rec_score: float = Field(..., description="Confidence score of the word recognition")
    det_score: float = Field(..., description="Confidence score of the word detection")


class TextDetectorSchema(BaseSchema):
    points: List[Quad] = Field(..., description="Detected text regions as quadrilaterals")
    scores: List[float] = Field(..., description="Confidence score per region")


class TextRecognizerSchema(BaseSchema):
    contents: List[str] = Field(..., description="Recognized text contents")
    directions: List[str] = Field(..., description="'horizontal' or 'vertical' per text")
    scores: List[float] = Field(..., description="Confidence score per text")
    points: List[Quad] = Field(..., description="Quadrilaterals of the recognized texts")


class OCRSchema(BaseSchema):
    words: List[WordPrediction] = Field(..., description="Recognized words")


Box = conlist(int, min_length=4, max_length=4)


class Element(BaseSchema):
    """One layout region (reference schemas/document_analyzer.py:9-29): what a layout analyzer returns per paragraph /
    figure."""
    id: Union[str, None] = Field(None, description="Unique identifier of the element")
    box: Box = Field(..., description="[x1, y1, x2, y2]")
    score: float = Field(..., description="Detection confidence")
    role: Union[str, None] = Field(..., description="e.g. 'section_headings', 'page_header', 'page_footer'")
    contents: Union[str, None] = Field(None, description="Text content of the element")


class ParagraphSchema(BaseSchema):
    box: Box
    contents: Union[str, None]
    direction: Union[str, None]
    order: Union[int, None]
    role: Union[str, None]


class TableCellSchema(BaseSchema):
    col: int
    row: int
    col_span: int
    row_span: int
    box: Box
    contents: Union[str, None]


class TableLineSchema(BaseSchema):
    box: Box
    score: float


class TableStructureRecognizerSchema(BaseSchema):
    """reference schemas/document_analyzer.py:94-118."""
    box: Box
    n_row: int
    n_col: int
    rows: List[TableLineSchema]
    cols: List[TableLineSchema]
    spans: List[TableLineSchema] = Field(default_factory=list)
    cells: List[TableCellSchema]
    order: int


class LayoutParserSchema(BaseSchema):
    """reference schemas/document_analyzer.py:183-186: what LayoutParser returns (tables are plain regions here)."""
    paragraphs: List[Element]
    tables: List[Element]
    figures: List[Element]


class LayoutAnalyzerSchema(BaseSchema):
    """What the layout half (reference layout_analyzer.py:38-49) hands to DocumentAnalyzer.aggregate."""
    paragraphs: List[Element]
    tables: List[TableStructureRecognizerSchema]
    figures: List[Element]


class FigureSchema(BaseSchema):
    box: Box
    order: Union[int, None]
    paragraphs: List[ParagraphSchema]
    direction: Union[str, None]
    figure_path: Union[str, None] = None


class DocumentAnalyzerSchema(BaseSchema):
    """reference DocumentAnalyzerSchema (schemas/document_analyzer.py:207-226).  Tables / figures / layout paragraphs
    come from a layout analyzer (the RT-DETRv2 models are outside this repo's hot path, SURVEY.md section 8f); without
    one every word becomes its own paragraph, exactly what the reference's aggregate does with an empty layout."""
    paragraphs: List[ParagraphSchema] = Field(default_factory=list)
    tables: List[TableStructureRecognizerSchema] = Field(default_factory=list)
    words: List[WordPrediction] = Field(default_factory=list)
    figures: List[FigureSchema] = Field(default_factory=list)


class CellSchema(BaseSchema):
    """One cell of a cell-detected table (reference schemas/table_semantic_parser.py:62-101).  row / col / spans and
    contents stay None until a table-semantic parser fills them."""
    meta: Dict[str, Any] = Field(default_factory=dict, description="Additional metadata for template/semantics")
    contents: Union[str, None] = Field(..., description="Text content of the cell")
    role: Union[str, None] = Field(..., description="Role of the cell, e.g., ['cell', 'header', 'empty', 'group']")
    id: Union[str, None] = Field(..., description="Unique identifier of the cell")
    box: Box = Field(..., description="Bounding box of the cell in the format [x1, y1, x2, y2]")
    row: Union[int, None] = Field(..., description="Row index of the cell in the table")
    col: Union[int, None] = Field(..., description="Column index of the cell in the table")
    row_span: Union[int, None] = Field(..., description="Number of rows spanned by the cell")
    col_span: Union[int, None] = Field(..., description="Number of columns spanned by the cell")


class RegionSchema(BaseSchema):
    """A region the cell detector predicts directly (kv_item / grid), reference :104-112."""
    id: Union[str, None] = Field(None, description="Region id")
    box: Box = Field(..., description="Bounding box [x1, y1, x2, y2]")
    role: str = Field(..., description="Region role, e.g., ['kv_item', 'grid']")
    score: float = Field(1.0, description="Detection score")


class TableDetectorSchema(BaseSchema):
    """What CellDetector returns per table (reference :115-140)."""
    id: Union[str, None] = Field(..., description="Unique identifier of the table")
    box: Box = Field(..., description="Bounding box of the table in the format [x1, y1, x2, y2]")
    role: Union[str, None] = Field(..., description="Role of the table region")
    cells: List[CellSchema] = Field(..., description="List of detected table cells")
    kv_regions: List[RegionSchema] = Field(default_factory=list, description="Model-predicted key-value item regions")
    grid_regions: List[RegionSchema] = Field(default_factory=list, description="Model-predicted grid regions")
