"""Generate the committed fixtures under tests/golden/ from a checkout of the QuantEcon
dynamic_factor_models project.  Usage:  python tests/golden/make_golden.py <checkout>

Writes
  hom_fac_1_panels.npz   output of the ingestion oracle (oracle/readin.py) on
                         <checkout>/data/hom_fac_1.xlsx for datatype :All and :Real
                         (the notebook's `dataset_all` / `dataset`, Stock_Watson.ipynb:160,180)
  hom_fac_1_sheets.tsv.xz  every cell of the Monthly and Quarterly sheets of that workbook, the
                         only sheets ingestion reads (see save_sheets); tests/test_ingest.py rebuilds
                         an .xlsx from it with write_xlsx
  notebook_tables.json   the numeric tables stored as cell outputs of Stock_Watson.ipynb
                         (Tables 2A, 2B, 2C, 3 (visible part), 4, 5) -- the reference's only
                         golden values (SURVEY.md section 4)
"""
import json, lzma, os, re, sys, zipfile
from xml.sax.saxutils import escape
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle.readin import readin_data  # noqa: E402
from oracle.xlsx_min import read_sheet  # noqa: E402

ANSI = re.compile(r"\x1b\[[0-9;]*m")

SHEETS = ("Monthly", "Quarterly")
_NS_MAIN = "http://schemas.openxmlformats.org/spreadsheetml/2006/main"
_NS_REL = "http://schemas.openxmlformats.org/officeDocument/2006/relationships"
_NS_PKG = "http://schemas.openxmlformats.org/package/2006/relationships"
_CT = "application/vnd.openxmlformats-officedocument.spreadsheetml"


def _col_letters(j):
    s = ""
    j += 1
    while j:
        j, m = divmod(j - 1, 26)
        s = chr(65 + m) + s
    return s


def write_xlsx(path, sheets):
    """Minimal .xlsx of {sheet name: 2-D list of float / str / None}.  Numbers are written in the shortest form
    that reads back to the same double; strings go to the shared-string table."""
    sst, sid = [], {}
    parts = []
    for grid in sheets.values():
        rows = []
        for i, row in enumerate(grid):
            cells = []
            for j, v in enumerate(row):
                ref = f"{_col_letters(j)}{i + 1}"
                if isinstance(v, str):
                    if v not in sid:
                        sid[v] = len(sst); sst.append(v)
                    cells.append(f'<c r="{ref}" t="s"><v>{sid[v]}</v></c>')
                elif v is not None:
                    cells.append(f'<c r="{ref}"><v>{float(v)!r}</v></c>')
            if cells:
                rows.append(f'<row r="{i + 1}">{"".join(cells)}</row>')
        parts.append(f'<worksheet xmlns="{_NS_MAIN}"><sheetData>{"".join(rows)}</sheetData></worksheet>')
    n = len(parts)
    head = '<?xml version="1.0" encoding="UTF-8" standalone="yes"?>\n'

    def put(name, text):                                  # fixed member times: the same sheets give the same bytes
        z.writestr(zipfile.ZipInfo(name, (1980, 1, 1, 0, 0, 0)), text, zipfile.ZIP_DEFLATED, 9)

    with zipfile.ZipFile(path, "w") as z:
        put("[Content_Types].xml", head + '<Types xmlns="http://schemas.openxmlformats.org/package/2006/content-types">'
            '<Default Extension="rels" ContentType="application/vnd.openxmlformats-package.relationships+xml"/>'
            '<Default Extension="xml" ContentType="application/xml"/>'
            f'<Override PartName="/xl/workbook.xml" ContentType="{_CT}.sheet.main+xml"/>'
            + "".join(f'<Override PartName="/xl/worksheets/sheet{i}.xml" ContentType="{_CT}.worksheet+xml"/>' for i in range(1, n + 1))
            + f'<Override PartName="/xl/sharedStrings.xml" ContentType="{_CT}.sharedStrings+xml"/></Types>')
        put("_rels/.rels", head + f'<Relationships xmlns="{_NS_PKG}">'
            f'<Relationship Id="rId1" Type="{_NS_REL}/officeDocument" Target="xl/workbook.xml"/></Relationships>')
        put("xl/workbook.xml", head + f'<workbook xmlns="{_NS_MAIN}" xmlns:r="{_NS_REL}"><sheets>'
            + "".join(f'<sheet name="{escape(s)}" sheetId="{i}" r:id="rId{i}"/>' for i, s in enumerate(sheets, 1))
            + "</sheets></workbook>")
        put("xl/_rels/workbook.xml.rels", head + f'<Relationships xmlns="{_NS_PKG}">'
            + "".join(f'<Relationship Id="rId{i}" Type="{_NS_REL}/worksheet" Target="worksheets/sheet{i}.xml"/>' for i in range(1, n + 1))
            + f'<Relationship Id="rId{n + 1}" Type="{_NS_REL}/sharedStrings" Target="sharedStrings.xml"/></Relationships>')
        for i, p in enumerate(parts, 1):
            put(f"xl/worksheets/sheet{i}.xml", head + p)
        put("xl/sharedStrings.xml", head + f'<sst xmlns="{_NS_MAIN}" count="{len(sst)}" uniqueCount="{len(sst)}">'
            + "".join(f'<si><t xml:space="preserve">{escape(s, {chr(13): "&#13;"})}</t></si>' for s in sst) + "</sst>")


def _enc(v):
    if isinstance(v, str):
        if "\t" in v or "\n" in v:
            raise ValueError(f"cell text {v!r} holds a tab or a newline")
        return "'" + v
    return "" if v is None else repr(float(v))


def _dec(c):
    return None if c == "" else c[1:] if c[0] == "'" else float(c)


def save_sheets(src, dst):
    """Store every cell of the sheets SHEETS of the workbook `src` (1.1 MB) in `dst`, losslessly, as xz-compressed
    text: per sheet a line "<name> <rows> <columns>" (tab-separated), then one line per column holding its cells
    separated by tabs -- empty for a blank cell, 'text for text, otherwise the shortest decimal form of the double.
    Column by column the numbers compress to about a quarter of the workbook."""
    lines = []
    for sheet in SHEETS:
        g = read_sheet(src, sheet)
        w = max(len(r) for r in g)
        lines.append(f"{sheet}\t{len(g)}\t{w}")
        lines += ["\t".join(_enc(r[j] if j < len(r) else None) for r in g) for j in range(w)]
    with open(dst, "wb") as f:
        f.write(lzma.compress("\n".join(lines).encode(), preset=9 | lzma.PRESET_EXTREME))


def load_sheets(path):
    """Inverse of save_sheets: {sheet name: 2-D list of float / str / None}."""
    with open(path, "rb") as f:
        lines = lzma.decompress(f.read()).decode().split("\n")
    out, k = {}, 0
    while k < len(lines):
        name, n, w = lines[k].split("\t")
        cols = [lines[k + 1 + j].split("\t") for j in range(int(w))]
        out[name] = [[_dec(c[i]) for c in cols] for i in range(int(n))]
        k += 1 + int(w)
    return out


def parse_millboard(text):
    rows = []
    for line in ANSI.sub("", text).splitlines():
        cells = [c.strip() for c in line.strip().strip("|").split("|")]
        try:
            vals = [float(c) for c in cells[1:]]
        except ValueError:
            continue
        if vals:
            rows.append(vals)
    return rows


def main(ref):
    xlsx = os.path.join(ref, "data", "hom_fac_1.xlsx")
    a = readin_data(xlsx, "All"); r = readin_data(xlsx, "Real")
    np.savez_compressed(os.path.join(HERE, "hom_fac_1_panels.npz"),
                        all_bpdata=a["bpdata"], all_inclcode=a["inclcode"], all_names=np.array(a["bpnamevec"]),
                        real_bpdata=r["bpdata"], real_inclcode=r["inclcode"], real_names=np.array(r["bpnamevec"]),
                        calds=np.array(a["calds"]))
    save_sheets(xlsx, os.path.join(HERE, "hom_fac_1_sheets.tsv.xz"))
    nb = json.load(open(os.path.join(ref, "Stock_Watson.ipynb")))
    outs = {}
    for i, c in enumerate(nb["cells"]):
        if c["cell_type"] != "code":
            continue
        txt = []
        for o in c.get("outputs", []):
            if "text" in o:
                txt.append("".join(o["text"]))
            elif "data" in o and "text/plain" in o["data"]:
                txt.append("".join(o["data"]["text/plain"]))
        outs[i] = txt
    tables = {}
    tables["table2A"] = parse_millboard(outs[35][0])      # cols: nfac, traceR2, margR2, BN-ICp2, AH-ER
    tables["table2B"] = parse_millboard(outs[37][0])
    tables["table2C"] = parse_millboard(outs[39][0])      # rows: n dynamic; cols: n dyn, then static 1..10
    # Table 3: 207x10 R2, visible: first 13 + last 12 rows, columns 1-3 and 8-10
    t3 = []
    for line in outs[55][0].splitlines()[1:]:
        toks = line.replace("…", " ").replace("⋱", " ").replace("⋮", " ").split()
        if len(toks) == 6:
            t3.append([float(x) for x in toks])
    tables["table3_visible"] = {"rows_head": 13, "rows_tail": 12, "cols": [1, 2, 3, 8, 9, 10], "values": t3}
    nums = lambda s: [[float(x) for x in ln.split()] for ln in s.splitlines()[1:] if ln.strip()]
    tables["table4"] = {"chow_qlr_r4": nums(outs[58][0]), "chow_qlr_r8": nums(outs[58][1]),
                        "cor_r4": nums(outs[58][2]), "cor_r8": nums(outs[58][3])}
    t5 = {}
    lines = outs[61][0].splitlines()
    for k in range(0, len(lines), 3):
        name = lines[k].split()[1]
        t5[name] = {"resid": [float(x) for x in lines[k + 1].strip("[]").split()],
                    "level": [float(x) for x in lines[k + 2].strip("[]").split()]}
    tables["table5"] = t5
    tables["source"] = "stored cell outputs of Stock_Watson.ipynb (Julia 1.0.2)"
    json.dump(tables, open(os.path.join(HERE, "notebook_tables.json"), "w"), indent=1)
    print({k: (len(v) if isinstance(v, list) else "...") for k, v in tables.items()})


if __name__ == "__main__":
    main(sys.argv[1])
