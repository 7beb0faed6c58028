"""CPU: the text front-end (auralis_b200/textnorm.py, text.py) against golden vectors produced by the reference's own
functions (tests/golden/text_cleaners.json, generator tests/golden/make_text_golden.py), and live against the reference
when /root/reference is mounted.  Number WORDS are third-party (num2words): both sides use the same marker function, so
what is pinned is everything the reference itself does around them."""
import json
import os

import pytest

from auralis_b200 import text as X
from auralis_b200 import textnorm as T
from oracle import ref_text

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "text_cleaners.json")


def _ours(rec):
    fn, lang, s = rec["fn"], rec["lang"], rec["in"]
    if fn == "expand_abbreviations_multilingual":
        return T.expand_abbreviations_multilingual(s, lang)
    if fn == "expand_symbols_multilingual":
        return T.expand_symbols_multilingual(s, lang)
    if fn == "expand_numbers_multilingual":
        return T.expand_numbers_multilingual(s, lang, n2w=ref_text.marker_num2words)
    if fn == "multilingual_cleaners":
        return T.multilingual_cleaners(s, lang, n2w=ref_text.marker_num2words)
    if fn == "basic_cleaners":
        return T.basic_cleaners(s)
    if fn == "split_sentence":
        return X.split_sentence(s, lang, rec["limit"])
    if fn == "find_best_split_point":
        return X.find_best_split_point(s, rec["limit"], 30)
    raise KeyError(fn)


def test_golden_vectors_from_the_reference():
    recs = json.load(open(GOLD, encoding="utf-8"))["records"]
    assert len(recs) >= 120
    seen = set()
    for rec in recs:
        assert _ours(rec) == rec["out"], (rec["fn"], rec["lang"], rec["in"][:60])
        seen.add((rec["fn"], rec["lang"]))
    # every cleaned language is covered by every table-driven stage
    for lang in ["en", "es", "fr", "de", "it", "pt", "pl", "ar", "zh", "cs", "ru", "nl", "tr", "hu", "ko"]:
        assert ("expand_abbreviations_multilingual", lang) in seen and ("expand_symbols_multilingual", lang) in seen
        assert ("expand_numbers_multilingual", lang) in seen and ("multilingual_cleaners", lang) in seen


def test_live_against_the_reference_module():
    """Random cleaner inputs and sentence splits; the reference tokenizer's answers are stored in
    tests/golden/text_reference_fuzz.npz (tests/reference_records.py)."""
    import random
    from reference_records import Records
    rec = Records("text_reference_fuzz")
    rng = random.Random(7)
    alphabet = "abc dr. mr. sr. st. co. 1 2 3 12 1.234 5,50 $ £ € % & # @ ° º ª th st er e . , ; ! ?".split(" ")
    for lang in ["en", "es", "fr", "de", "it", "pt", "pl", "ar", "zh", "cs", "ru", "nl", "tr", "hu", "ko"]:
        for _ in range(60):
            s = " ".join(rng.choice(alphabet) for _ in range(rng.randint(1, 14)))
            if rng.random() < 0.5:
                s = s.replace(" ", "", rng.randint(0, 4))
            want = rec(f"multilingual_cleaners[{lang}]{s}", lambda: ref_text.load().multilingual_cleaners(s, lang))
            assert T.multilingual_cleaners(s, lang, n2w=ref_text.marker_num2words) == want, (lang, s)
    for _ in range(20):
        n = rng.randint(3, 30)
        s = " ".join(rng.choice(["Short one.", "A somewhat longer sentence, with a clause; and more - much more - to say about it all", "Why?",
                                 "Numbers like 1.5 do not end sentences.", "Ellipsis... then more!"]) for _ in range(n))
        lim = rng.choice([40, 82, 166, 250])
        assert X.split_sentence(s, "en", lim) == rec(f"split_sentence[{lim}]{s}", lambda: ref_text.load().split_sentence(s, "en", lim))


def test_number_words_follow_num2words_conventions():
    """Word lists restated from num2words' published conventions (no copy of num2words to compare with: unpinned)."""
    v = T.verbalise
    assert v(0) == "zero" and v(21) == "twenty-one" and v(110) == "one hundred and ten" and v(1001) == "one thousand and one"
    assert v(1234) == "one thousand, two hundred and thirty-four" and v(1200000) == "one million, two hundred thousand"
    assert v(1000001) == "one million and one"
    assert v(1, ordinal=True) == "first" and v(12, ordinal=True) == "twelfth" and v(21, ordinal=True) == "twenty-first"
    assert v(100, ordinal=True) == "one hundredth" and v(43, ordinal=True) == "forty-third"
    assert v(3.05) == "three point zero five" and v(1.10) == "one point one"
    assert v(5.5, to="currency", currency="USD") == "five dollars, fifty cents"
    assert v(2.01, to="currency", currency="GBP") == "two pounds, one penny"
    # Spanish
    assert [v(n, lang="es") for n in (16, 21, 22, 31, 100, 101, 500, 1000, 2000, 21000, 1000000, 2000000)] == [
        "dieciséis", "veintiuno", "veintidós", "treinta y uno", "cien", "ciento uno", "quinientos", "mil", "dos mil",
        "veintiún mil", "un millón", "dos millones"]
    assert v(3.14, lang="es") == "tres punto uno cuatro" and v(1, ordinal=True, lang="es") == "primero"
    assert v(13, ordinal=True, lang="es") == "decimotercero" and v(21, ordinal=True, lang="es") == "vigésimo primero"
    assert v(1.5, to="currency", currency="EUR", lang="es") == "un euro con cincuenta céntimos"
    # French
    assert [v(n, lang="fr") for n in (17, 21, 70, 71, 80, 81, 90, 99, 100, 200, 201, 1000, 2000, 80000, 1000000)] == [
        "dix-sept", "vingt et un", "soixante-dix", "soixante et onze", "quatre-vingts", "quatre-vingt-un", "quatre-vingt-dix",
        "quatre-vingt-dix-neuf", "cent", "deux cents", "deux cent un", "mille", "deux mille", "quatre-vingt mille", "un million"]
    assert v(2.5, lang="fr") == "deux virgule cinq" and v(1, ordinal=True, lang="fr") == "premier"
    assert v(2, ordinal=True, lang="fr") == "deuxième" and v(5, ordinal=True, lang="fr") == "cinquième"
    assert v(9, ordinal=True, lang="fr") == "neuvième" and v(21, ordinal=True, lang="fr") == "vingt et unième"
    assert v(80, ordinal=True, lang="fr") == "quatre-vingtième"
    assert v(5.5, to="currency", currency="EUR", lang="fr") == "cinq euros et cinquante centimes"
    # German
    assert [v(n, lang="de") for n in (1, 16, 21, 30, 100, 101, 121, 1000, 1001, 2000, 1000000, 2000000, 1000001)] == [
        "eins", "sechzehn", "einundzwanzig", "dreißig", "einhundert", "einhunderteins", "einhunderteinundzwanzig", "eintausend",
        "eintausendeins", "zweitausend", "eine million", "zwei millionen", "eine million eins"]
    assert v(3.14, lang="de") == "drei komma eins vier"
    assert [v(n, ordinal=True, lang="de") for n in (1, 3, 7, 8, 19, 20, 21, 101)] == [
        "erste", "dritte", "siebte", "achte", "neunzehnte", "zwanzigste", "einundzwanzigste", "einhunderterste"]
    assert v(1.5, to="currency", currency="EUR", lang="de") == "ein euro und fünfzig cent"
    # Italian
    assert [v(n, lang="it") for n in (21, 23, 28, 33, 100, 101, 180, 200, 1000, 1234, 2000, 1000000, 2000000)] == [
        "ventuno", "ventitré", "ventotto", "trentatré", "cento", "centouno", "centottanta", "duecento", "mille",
        "milleduecentotrentaquattro", "duemila", "un milione", "due milioni"]
    assert v(2.75, lang="it") == "due virgola sette cinque" and v(3, ordinal=True, lang="it") == "terzo"
    assert v(11, ordinal=True, lang="it") == "undicesimo" and v(23, ordinal=True, lang="it") == "ventitreesimo"
    assert v(5.5, to="currency", currency="EUR", lang="it") == "cinque euro e cinquanta centesimi"
    # Portuguese (European)
    assert [v(n, lang="pt") for n in (16, 21, 100, 101, 200, 1000, 1001, 1100, 1234, 2000, 1000000, 2000000)] == [
        "dezasseis", "vinte e um", "cem", "cento e um", "duzentos", "mil", "mil e um", "mil e cem",
        "mil duzentos e trinta e quatro", "dois mil", "um milhão", "dois milhões"]
    assert v(1.5, lang="pt") == "um vírgula cinco" and v(11, ordinal=True, lang="pt") == "décimo primeiro"
    assert v(5.5, to="currency", currency="EUR", lang="pt") == "cinco euros e cinquenta cêntimos"
    # Dutch, Turkish, Hungarian, Russian, Polish, Czech (numwords_more.py)
    assert [v(n, lang="nl") for n in (0, 21, 22, 23, 100, 101, 1000, 1234, 2000, 21000, 1000000, 2500000)] == [
        "nul", "eenentwintig", "tweeëntwintig", "drieëntwintig", "honderd", "honderdeen", "duizend", "duizendtweehonderdvierendertig",
        "tweeduizend", "eenentwintigduizend", "een miljoen", "twee miljoen vijfhonderdduizend"]
    assert [v(n, ordinal=True, lang="nl") for n in (1, 3, 8, 13, 20, 100, 101)] == [
        "eerste", "derde", "achtste", "dertiende", "twintigste", "honderdste", "honderdeerste"]
    assert v(3.25, lang="nl") == "drie komma twee vijf"
    assert [v(n, lang="tr") for n in (0, 11, 100, 101, 1000, 2345, 1000000)] == [
        "sıfır", "onbir", "yüz", "yüzbir", "bin", "ikibinüçyüzkırkbeş", "birmilyon"]
    assert [v(n, ordinal=True, lang="tr") for n in (1, 4, 6, 9, 20, 34, 100)] == [
        "birinci", "dördüncü", "altıncı", "dokuzuncu", "yirminci", "otuzdördüncü", "yüzüncü"]
    assert [v(n, lang="hu") for n in (0, 2, 12, 21, 200, 1000, 1999, 2000, 2001, 22000, 2500000)] == [
        "nulla", "kettő", "tizenkettő", "huszonegy", "kétszáz", "ezer", "ezerkilencszázkilencvenkilenc", "kétezer", "kétezer-egy",
        "huszonkétezer", "kétmillió-ötszázezer"]
    assert v(3.5, lang="hu") == "három egész öt tized"
    assert [v(n, ordinal=True, lang="hu") for n in (1, 2, 3, 5, 10, 11, 12, 20, 21, 36, 100, 101, 1000, 2001)] == [
        "első", "második", "harmadik", "ötödik", "tizedik", "tizenegyedik", "tizenkettedik", "huszadik", "huszonegyedik",
        "harminchatodik", "századik", "százegyedik", "ezredik", "kétezer-egyedik"]
    assert [v(n, lang="ru") for n in (0, 21, 101, 1000, 2000, 5000, 11000, 21000, 1000000, 2000000, 5000000)] == [
        "ноль", "двадцать один", "сто один", "одна тысяча", "две тысячи", "пять тысяч", "одиннадцать тысяч", "двадцать одна тысяча",
        "один миллион", "два миллиона", "пять миллионов"]
    assert v(3.05, lang="ru") == "три запятая ноль пять"
    assert [v(n, ordinal=True, lang="ru") for n in (1, 3, 11, 21, 40, 100, 121, 1000, 2000)] == [
        "первый", "третий", "одиннадцатый", "двадцать первый", "сороковой", "сотый", "сто двадцать первый", "тысячный", "двухтысячный"]
    assert [v(n, lang="pl") for n in (0, 21, 1000, 2000, 5000, 12000, 22000, 1000000)] == [
        "zero", "dwadzieścia jeden", "tysiąc", "dwa tysiące", "pięć tysięcy", "dwanaście tysięcy", "dwadzieścia dwa tysiące", "milion"]
    assert v(3.25, lang="pl") == "trzy przecinek dwadzieścia pięć"
    assert [v(n, lang="cz") for n in (0, 21, 200, 1000, 2000, 5000)] == ["nula", "dvacet jedna", "dvě stě", "tisíc", "dva tisíce", "pět tisíc"]
    assert v(5.5, to="currency", currency="EUR", lang="nl") == "vijf euro, vijftig cent"
    assert v(21.05, to="currency", currency="USD", lang="ru") == "двадцать один доллар, пять центов"
    assert v(2.5, to="currency", currency="EUR", lang="pl") == "dwa euro, pięćdziesiąt centów"
    assert v(5.22, to="currency", currency="USD", lang="cz") == "pět dolarů, dvacet dva centy"
    # what is not restated keeps its digits: Arabic and Korean altogether, ordinals of pl / cs
    assert v(12, lang="ar") == "12" and v(7, ordinal=True, lang="cz") == "7"


def test_number_words_are_injective_and_clean():
    """A table typo shows up as two numbers with one reading, an empty group or a stray digit: every restated language must
    give 30 000 consecutive integers (and a few large ones) distinct, trimmed, digit-free readings."""
    v = T.verbalise
    probe = list(range(0, 30001, 1)) + [10 ** 6, 10 ** 6 + 1, 2 * 10 ** 6 + 345678, 10 ** 9, 123456789012]
    for lang in ("en", "es", "fr", "de", "it", "pt", "nl", "tr", "hu", "ru", "pl", "cs"):
        seen = {}
        for n in probe:
            w = v(n, lang=lang)
            assert w and w == w.strip() and "  " not in w and not any(ch.isdigit() for ch in w), (lang, n, w)
            assert w not in seen, (lang, n, seen[w], w)
            seen[w] = n


def test_long_digit_strings_never_raise():
    """Ids and phone numbers are digit strings too: every cleaned language must read them somehow (beyond their scale tables
    the six languages of numwords_more.py go digit by digit), never raise."""
    for lang in ("en", "es", "fr", "de", "it", "pt", "nl", "tr", "hu", "ru", "pl", "cs", "ar", "ko"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out = T.preprocess_text("id 123456789012345678901234567890, 999999999999999 and 1000000000000000.", lang)
        assert out and "  " not in out
    assert T.verbalise(10 ** 15, lang="ru") == "один ноль ноль ноль ноль ноль ноль ноль ноль ноль ноль ноль ноль ноль ноль ноль"
    assert T.verbalise(10 ** 15 - 1, lang="pl").startswith("dziewięćset dziewięćdziesiąt dziewięć bilionów")


def test_cleaners_end_to_end_with_number_words():
    c = T.preprocess_text('Dr. Smith paid $5.50 for the 21st "copy", 1,234 in all & 3.5% more.', "en")
    assert c == ("doctor smith paid five dollars, fifty cents for the twenty-first copy, one thousand, two hundred and "
                 "thirty-four in all and three point five percent more.")
    assert T.preprocess_text("Das  kostet 1.234 Euro & 20€", "de") == "das kostet eintausendzweihundertvierunddreißig euro und zwanzig euro"
    assert T.preprocess_text("El Sr. García pagó 20€ el 1º", "es") == "el señor garcía pagó veinte euros el primero"
    assert T.preprocess_text("Mme. Dupont a 71 ans & 2,5 chats", "fr") == "madame dupont a soixante et onze ans et deux virgule cinq chats"
    assert T.preprocess_text("ÇOK  İYİ", "tr") == "çok iyi"                                    # dotted capital İ mapped before lower()
    assert T.preprocess_text("To jest 12 & 3", "pl") == "to jest dwanaście i trzy"
    assert T.preprocess_text("Ik heb 21 appels en 3,5 liter op de 3de dag", "nl") == "ik heb eenentwintig appels en drie komma vijf liter op de derde dag"
    assert T.preprocess_text("У меня 21000 рублей", "ru") == "у меня двадцать одна тысяча рублей"
    assert T.preprocess_text("Het kost 20€ of $5,50.", "nl") == "het kost twintig euro of vijf dollar, vijftig cent."
    assert T.preprocess_text("Ez 20€ meg 1$.", "hu") == "ez húsz euró meg egy dollár."
    assert T.preprocess_text("هذا 12", "ar") == "هذا 12"                                        # digits kept (no Arabic number words)
    assert T.format_for_bpe("Hello there", "en") == "[en]hello[SPACE]there"
    assert T.format_for_bpe("你好", "zh-cn").startswith("[zh-cn]")
    assert T.preprocess_text("MiXed   Case", "xx") == "mixed case"


def test_romanisation_hooks_follow_the_reference_wiring(monkeypatch):
    """zh/ko/ja: the third-party romanisers are called the way tokenizer.py:727-739 calls them when present; absent -> warning."""
    import sys
    import types
    import warnings
    T._TRANSLIT_CACHE.clear(); T._TRANSLIT_WARNED.clear()
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        assert T.preprocess_text("你好 20%", "zh-cn") == "你好 百分之二十"              # cleaners still run; no pypinyin here
        assert T.preprocess_text("こんにちは", "ja") == "こんにちは"
    assert any("pypinyin" in str(x.message) for x in w) and any("cutlet" in str(x.message) for x in w)
    calls = {}
    pyp = types.ModuleType("pypinyin")
    pyp.Style = types.SimpleNamespace(TONE3="T3")

    def pinyin(text, style=None, heteronym=None, neutral_tone_with_five=None):
        calls["zh"] = (style, heteronym, neutral_tone_with_five)
        return [[f"<{ch}>"] for ch in text]
    pyp.pinyin = pinyin
    cut = types.ModuleType("cutlet")
    cut.Cutlet = lambda: types.SimpleNamespace(romaji=lambda t: "Konnichiwa")
    monkeypatch.setitem(sys.modules, "pypinyin", pyp)
    monkeypatch.setitem(sys.modules, "cutlet", cut)
    T._TRANSLIT_CACHE.clear()
    assert T.preprocess_text("你好", "zh") == "<你><好>" and calls["zh"] == ("T3", False, True)
    assert T.preprocess_text("こんにちは", "ja") == "konnichiwa"
    T._TRANSLIT_CACHE.clear(); T._TRANSLIT_WARNED.clear()
