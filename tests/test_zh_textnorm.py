"""CPU: the Chinese normaliser (auralis_b200/zh_textnorm.py) against the reference's own `zh_num2words` — golden records,
and a fuzz whose reference answers are stored in tests/golden/zh_textnorm_fuzz.npz (tests/reference_records.py)."""
import json
import os

from auralis_b200 import textnorm as T
from auralis_b200 import zh_textnorm as Z
from reference_records import Records
from zh_fixture import load_reference_zh, sentences

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "zh_textnorm.json")


def test_golden_records_from_the_reference():
    rec = json.load(open(GOLD, encoding="utf-8"))
    assert len(rec["sentences"]) >= 400 and len(rec["numbers"]) >= 150
    for r in rec["sentences"]:
        assert Z.normalize(r["in"]) == r["out"], r["in"]
    for r in rec["numbers"]:
        assert Z.num2chn(r["in"]) == r["cardinal"], r["in"]
        assert Z.num2chn(r["in"], alt_two=False, use_units=False) == r["digits"], r["in"]


def test_examples():
    assert Z.normalize("我有2个苹果和12.5%的股份") == "我有二个苹果和百分之十二点五的股份"
    assert Z.normalize("2023年10月5日，价格是3.50元") == "二零二三年十月五日,价格是三点五零元"
    assert Z.normalize("电话13812345678或010-12345678") == "电话一三八一二三四五六七八或零一零一二三四五六七八"
    assert Z.normalize("1/3的人 202 10500 P2P") == "三分之一的人 两百零二 一零五零零 P2P"
    # through the cleaner pipeline: lowercase, zh numbers + punctuation, zh symbol words, whitespace
    assert T.multilingual_cleaners("价格 5£ 和 3°, 共12个!", "zh") == "价格 五 英镑 和 三 度 , 共十二个,"


def test_live_fuzz_against_the_reference_module():
    rec = Records("zh_textnorm_fuzz")
    fuzz = sentences(3000, 99)
    want = rec("TextNorm", lambda: [load_reference_zh().TextNorm()(s) for s in fuzz])
    for s, w in zip(fuzz, want, strict=True):
        assert Z.normalize(s) == w, s

    def reference_cleaners(ss):
        from oracle import ref_text
        ref_tok = ref_text.load()
        return [ref_tok.multilingual_cleaners(s, "zh") for s in ss]
    fuzz = sentences(300, 7)                       # the whole zh cleaner chain of the reference tokenizer
    want = rec("multilingual_cleaners", lambda: reference_cleaners(fuzz))
    for s, w in zip(fuzz, want, strict=True):
        assert T.multilingual_cleaners(s, "zh") == w, s
