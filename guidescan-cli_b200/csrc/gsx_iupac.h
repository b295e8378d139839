// gsx_iupac.h -- IUPAC class letters in PAMs: the one table of members, complements and expansion shared by the search's PAM
// preparation (gsx_api.cpp), the k-mer generator (gsx_kmers.cu), the decoder (gsx_decode.cu) and the SAM formatter.
//
// A PAM character is one of A, C, G, T, N or a class letter R={A,G} Y={C,T} S={C,G} W={A,T} K={G,T} M={A,C} B={C,G,T} D={A,G,T}
// H={A,C,T} V={A,C,G} (upper case only).  A class matches a genome base that is one of its members, at no mismatch cost, like N;
// unlike N it never matches a literal genome N or any other non-ACGT character.
#ifndef GSX_IUPAC_H
#define GSX_IUPAC_H
#include "gsx_types.h"
#include <deque>
#include <string>
#include <vector>

namespace gsx {

// member mask of a PAM letter (A=1, C=2, G=4, T=8; N=15); 0 = not a PAM letter
GSX_HD uint32_t iupac_mask(char c) {
    switch (c) {
    case 'A': return 1u; case 'C': return 2u; case 'G': return 4u; case 'T': return 8u;
    case 'R': return 5u; case 'Y': return 10u; case 'S': return 6u; case 'W': return 9u; case 'K': return 12u; case 'M': return 3u;
    case 'B': return 14u; case 'D': return 13u; case 'H': return 11u; case 'V': return 7u;
    case 'N': return 15u;
    default: return 0u;
    }
}
// a class letter: two or three members (not A, C, G, T or N)
GSX_HD bool iupac_is_class(char c) { const uint32_t m = iupac_mask(c); return m != 0u && m != 15u && (m & (m - 1u)) != 0u; }
GSX_HD bool iupac_pam_char(char c) { return iupac_mask(c) != 0u; }
// bit of a genome base (A=1, C=2, G=4, T=8); 0 for N and any other character
GSX_HD uint32_t iupac_base_bit(char c) { return c == 'A' ? 1u : c == 'C' ? 2u : c == 'G' ? 4u : c == 'T' ? 8u : 0u; }
// does PAM letter p accept the genome character s?  N accepts everything (a literal genome N included), a class its members
GSX_HD bool iupac_pam_fits(char p, char s) { return p == 'N' || p == s || (iupac_is_class(p) && (iupac_mask(p) & iupac_base_bit(s)) != 0u); }
// complement of a PAM letter: R<->Y, K<->M, B<->V, D<->H, S, W and N to themselves, A<->T, C<->G; any other character unchanged
GSX_HD char iupac_complement(char c) {
    switch (c) {
    case 'A': return 'T'; case 'T': return 'A'; case 'C': return 'G'; case 'G': return 'C';
    case 'R': return 'Y'; case 'Y': return 'R'; case 'K': return 'M'; case 'M': return 'K';
    case 'B': return 'V'; case 'V': return 'B'; case 'D': return 'H'; case 'H': return 'D';
    default: return c;
    }
}

// Every concrete PAM a pattern stands for, as the reference's generate_kmers.py expands N: breadth first, the first expandable
// letter (N or a class) first, its members in the order A, C, T, G.  For an A/C/G/T/N pattern this is generate_kmers.py's list.
inline std::vector<std::string> iupac_expand(const std::string& pam) {
    std::deque<std::string> q{pam};
    auto expandable = [](const std::string& s) { for (size_t i = 0; i < s.size(); i++) if (s[i] == 'N' || iupac_is_class(s[i])) return i; return std::string::npos; };
    auto any = [&]() { for (auto& s : q) if (expandable(s) != std::string::npos) return true; return false; };
    while (any()) {
        std::string s = q.front(); q.pop_front();
        const size_t at = expandable(s);
        if (at == std::string::npos) { q.push_back(s); continue; }
        const uint32_t m = iupac_mask(s[at]);
        for (char c : {'A', 'C', 'T', 'G'}) if (m & iupac_base_bit(c)) { std::string t = s; t[at] = c; q.push_back(t); }
    }
    return std::vector<std::string>(q.begin(), q.end());
}
// class letters (not N) expanded into their members, N kept: the concrete PAM list a class PAM is equivalent to in a search
inline std::vector<std::string> iupac_expand_classes(const std::string& pam) {
    std::vector<std::string> out{std::string()};
    for (char c : pam) {
        std::vector<std::string> nxt;
        for (const std::string& s : out) {
            if (!iupac_is_class(c)) { nxt.push_back(s + c); continue; }
            for (char b : {'A', 'C', 'G', 'T'}) if (iupac_mask(c) & iupac_base_bit(b)) nxt.push_back(s + b);
        }
        out.swap(nxt);
    }
    return out;
}

}  // namespace gsx
#endif
