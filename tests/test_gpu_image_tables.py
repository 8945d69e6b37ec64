"""Which optional tables an index image holds under each table knob (the knob table above plan_tables in csrc/fmb_lib.cu), on the DNA
layout (bidirectional and unidirectional) and on the generic layout; and that an index created from the exported BWT and samples
(fmb_index_create_ex, which fmb_index_load uses) holds the same tables in the same number of bytes as the index built from the text."""
import pytest

from test_gpu_extract import collection

pytestmark = pytest.mark.gpu

# the knob set for one column (FMB_KMER_K=0 sizes the exact-search k-mer table to nothing), then info.tables per index for each column:
# FMB_TABLE_PAIR 1, KMER 2, JUMP 4, JUMP_REV 8, LOCBLOCK 16, LOCROW 32, BIKMER 64, JUMP4 128, JUMP32 256
KNOBS = [None, ("FMB_NO_JUMP", "1"), ("FMB_NO_JUMP32", "1"), ("FMB_NO_JUMP4", "1"), ("FMB_NO_BIKMER", "1"), ("FMB_NO_LOCBLOCKS", "1"),
         ("FMB_NO_LOCROW", "1"), ("FMB_KMER_K", "0")]
TABLES = {
    (5, True): [511, 115, 255, 383, 447, 463, 479, 509],
    (5, False): [439, 51, 183, 311, 439, 391, 407, 437],
    (21, True): [224, 96, 224, 224, 160, 224, 192, 224],       # generic layout: the bidirectional k-mer table gets k = 3 at ~1 M symbols
}


@pytest.fixture(scope="module")
def texts(gpu):
    return {sigma: collection(sigma, 40, 3, min_len=1, max_len=50_000)[1] for sigma in (5, 21)}


@pytest.mark.parametrize("sigma,bidirectional", list(TABLES))
@pytest.mark.parametrize("column", range(len(KNOBS)), ids=[k[0] if k else "none" for k in KNOBS])
def test_knob_tables_and_constructors(gpu, texts, monkeypatch, sigma, bidirectional, column):
    if KNOBS[column]:
        monkeypatch.setenv(*KNOBS[column])               # read when an index is planned, by both constructors
    built = gpu.Index.build(sigma, texts[sigma], sampling_rate=16, bidirectional=bidirectional)
    created = gpu.Index.from_bwt(sigma, *built.export())
    assert built.info.tables == TABLES[(sigma, bidirectional)][column]
    assert created.info.tables == built.info.tables
    assert created.info.device_bytes == built.info.device_bytes
