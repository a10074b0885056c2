// pcd_io.hpp -- ROS/PCL-free PCD v0.7 reader (ASCII, binary, binary_compressed) for the CLI harness.
// Same semantics as pcl::io::loadPCDFile as used by the reference client (src/calc_grasppoints_action_client.cpp:141):
// exactly POINTS records (extra ASCII lines ignored), tokens parsed straight to float (strtof),
// binary_compressed = uint32 compressed size, uint32 uncompressed size, LZF stream, fields stored struct-of-arrays.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <sstream>
#include <string>
#include <vector>

namespace hafpcd {

inline bool lzf_decompress(const unsigned char* ip, size_t in_len, unsigned char* out, size_t out_len) {
    size_t i = 0, o = 0;
    while (i < in_len) {
        unsigned ctrl = ip[i++];
        if (ctrl < 32) {
            size_t n = ctrl + 1;
            if (o + n > out_len || i + n > in_len) return false;
            memcpy(out + o, ip + i, n);
            i += n; o += n;
        } else {
            size_t len = ctrl >> 5;
            if (len == 7) { if (i >= in_len) return false; len += ip[i++]; }
            if (i >= in_len) return false;
            size_t dist = ((ctrl & 0x1f) << 8) + ip[i++] + 1;
            len += 2;
            if (dist > o || o + len > out_len) return false;
            for (size_t k = 0; k < len; k++, o++) out[o] = out[o - dist];
        }
    }
    return o == out_len;
}

// The tokens of one line of an ASCII DATA section: fields are separated by runs of blank, tab and CR only (PCL's boost::split
// on "\t\r "); vertical tab and form feed are token characters, as on the device (csrc/pcd_ingest.cuh, is_blank).
inline void ascii_tokens(const std::string& line, std::vector<std::string>& toks) {
    size_t p = 0;
    const size_t n = line.size();
    while (p < n) {
        while (p < n && (line[p] == ' ' || line[p] == '\t' || line[p] == '\r')) p++;
        size_t e = p;
        while (e < n && line[e] != ' ' && line[e] != '\t' && line[e] != '\r') e++;
        if (e > p) toks.push_back(line.substr(p, e - p));
        p = e;
    }
}
// A FLOAT32 token: strtof of its longest numeric prefix.  strtof would skip a leading vertical tab or form feed; those are
// token characters here, so such a token has no numeric prefix and reads 0, as on the device.
inline float ascii_token_value(const std::string& tok) {
    if (!tok.empty() && (tok[0] == '\v' || tok[0] == '\f')) return 0.0f;
    return strtof(tok.c_str(), NULL);
}

// The text header of a PCD v0.7 file, up to and including its DATA line (what pcl::PCDReader::readHeader takes from it for
// an xyz cloud).  Also used by the device ingest (csrc/pcd_ingest.cuh, haf_pcd_decode): the header stays host-side text.
struct PcdHeader {
    std::vector<std::string> fields, types;
    std::vector<int> sizes, counts;
    long npts = -1, width = 0, height = 1;
    std::string data_kind;     // "ascii" | "binary" | "binary_compressed"
    size_t data_begin = 0;     // offset of the first byte after the DATA line
    int idx[3] = {-1, -1, -1}; // field numbers of x, y, z
};
inline bool parse_pcd_header(const unsigned char* raw, size_t n_bytes, PcdHeader& h, std::string* err) {
    size_t pos = 0;
    while (pos < n_bytes) {
        size_t nl = pos;
        while (nl < n_bytes && raw[nl] != '\n') nl++;
        std::string line((const char*)&raw[pos], nl - pos);
        pos = nl + 1;
        if (line.empty() || line[0] == '#') continue;
        std::istringstream ss(line);
        std::string key;
        ss >> key;
        std::string tok;
        if (key == "FIELDS") while (ss >> tok) h.fields.push_back(tok);
        else if (key == "SIZE") while (ss >> tok) h.sizes.push_back(atoi(tok.c_str()));
        else if (key == "TYPE") while (ss >> tok) h.types.push_back(tok);
        else if (key == "COUNT") while (ss >> tok) h.counts.push_back(atoi(tok.c_str()));
        else if (key == "WIDTH") ss >> h.width;
        else if (key == "HEIGHT") ss >> h.height;
        else if (key == "POINTS") ss >> h.npts;
        else if (key == "DATA") { ss >> h.data_kind; break; }
    }
    h.data_begin = pos < n_bytes ? pos : n_bytes;
    if (h.npts < 0) h.npts = h.width * h.height;
    if (h.counts.empty()) h.counts.assign(h.fields.size(), 1);
    for (size_t k = 0; k < h.fields.size(); k++) { if (h.fields[k] == "x") h.idx[0] = (int)k; if (h.fields[k] == "y") h.idx[1] = (int)k; if (h.fields[k] == "z") h.idx[2] = (int)k; }
    if (h.idx[0] < 0 || h.idx[1] < 0 || h.idx[2] < 0 || h.sizes.size() != h.fields.size() || h.types.size() != h.fields.size() ||
        h.counts.size() != h.fields.size()) { if (err) *err = "PCD header lacks x/y/z fields"; return false; }
    if (h.npts < 0) { if (err) *err = "PCD header: negative point count"; return false; }
    return true;
}

// xyz: packed x,y,z floats.  Returns false with *err set on failure.
inline bool read_pcd(const std::string& path, std::vector<float>& xyz, std::string* err) {
    FILE* fp = fopen(path.c_str(), "rb");
    if (!fp) { if (err) *err = "cannot open " + path; return false; }
    std::vector<unsigned char> raw;
    unsigned char buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, fp)) > 0) raw.insert(raw.end(), buf, buf + n);
    fclose(fp);
    PcdHeader hd;
    if (!parse_pcd_header(raw.data(), raw.size(), hd, err)) return false;
    size_t pos = hd.data_begin;
    const std::vector<std::string>&fields = hd.fields, &types = hd.types;
    const std::vector<int>&sizes = hd.sizes, &counts = hd.counts;
    const long npts = hd.npts;
    const std::string& data_kind = hd.data_kind;
    xyz.assign((size_t)npts * 3, 0.0f);
    const int idx[3] = {hd.idx[0], hd.idx[1], hd.idx[2]};
    if (data_kind == "ascii") {
        std::vector<int> tokoff(fields.size() + 1, 0);
        for (size_t k = 0; k < fields.size(); k++) tokoff[k + 1] = tokoff[k] + counts[k];
        long rec = 0;
        while (pos < raw.size() && rec < npts) {
            size_t nl = pos;
            while (nl < raw.size() && raw[nl] != '\n') nl++;
            std::string line((const char*)&raw[pos], nl - pos);
            pos = nl + 1;
            std::vector<std::string> toks;
            ascii_tokens(line, toks);
            if (toks.empty()) continue;
            for (int a = 0; a < 3; a++) {
                if (tokoff[idx[a]] >= (int)toks.size()) { if (err) *err = "short ASCII record in " + path; return false; }
                xyz[rec * 3 + a] = ascii_token_value(toks[tokoff[idx[a]]]);
            }
            rec++;
        }
        if (rec != npts) { if (err) *err = "fewer records than POINTS in " + path; return false; }
        return true;
    }
    for (int a = 0; a < 3; a++) if (types[idx[a]] != "F" || sizes[idx[a]] != 4) { if (err) *err = "x/y/z must be float32"; return false; }
    if (data_kind == "binary") {
        size_t rec_bytes = 0;
        std::vector<size_t> foff(fields.size());
        for (size_t k = 0; k < fields.size(); k++) { foff[k] = rec_bytes; rec_bytes += (size_t)sizes[k] * counts[k]; }
        if (pos + rec_bytes * npts > raw.size()) { if (err) *err = "binary PCD truncated"; return false; }
        for (long r = 0; r < npts; r++)
            for (int a = 0; a < 3; a++) memcpy(&xyz[r * 3 + a], &raw[pos + r * rec_bytes + foff[idx[a]]], 4);
        return true;
    }
    if (data_kind == "binary_compressed") {
        if (pos + 8 > raw.size()) { if (err) *err = "compressed PCD truncated"; return false; }
        uint32_t comp, uncomp;
        memcpy(&comp, &raw[pos], 4);
        memcpy(&uncomp, &raw[pos + 4], 4);
        if (pos + 8 + comp > raw.size()) { if (err) *err = "compressed PCD truncated"; return false; }
        std::vector<unsigned char> blob(uncomp);
        if (!lzf_decompress(&raw[pos + 8], comp, blob.data(), uncomp)) { if (err) *err = "corrupt LZF stream in " + path; return false; }
        std::vector<size_t> foff(fields.size());
        size_t off = 0;
        for (size_t k = 0; k < fields.size(); k++) { foff[k] = off; off += (size_t)npts * sizes[k] * counts[k]; }
        for (int a = 0; a < 3; a++)
            for (long r = 0; r < npts; r++) memcpy(&xyz[r * 3 + a], &blob[foff[idx[a]] + (size_t)r * 4 * counts[idx[a]]], 4);
        return true;
    }
    if (err) *err = "unsupported PCD DATA kind " + data_kind;
    return false;
}

}  // namespace hafpcd
