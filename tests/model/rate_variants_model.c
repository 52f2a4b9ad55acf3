/* CPU model of the parallel rate loop (k_enc_probe + k_enc_resolve in csrc/m3s_encode.cu), run against the oracle's own
 * sequential iteration loop.  TEST INFRASTRUCTURE (tests/test_rate_variants_model.py builds and runs it); it includes the oracle.
 *
 * Claim under test: a granule's rate-loop result depends on its predecessors only through (a) the <= 3 payload bits at its
 * hide_str_offset -- one of 15 variants -- and (b) the slot's stale address1..3, and (b) only when a probe finds big_values == 0
 * among non-zero values before any probe of the same walk had big values.  So every variant can be evaluated without the chain
 * ("probe"), and a sequential pass that only looks results up ("resolve", redoing the flagged granules with the true state)
 * reproduces the reference's side info, step sizes, addresses and hide_str_offset exactly.
 *
 * usage: rate_variants_model pcm.raw n_frames bitrate_kbps payload.txt [payload_len|-1 [sample_rate]]
 *   ->  "granules N silent S slow R bad B maxsteps M"
 * (bad = granules where the model and the oracle disagree; must be 0.  maxsteps = the most distinct steps the active variants of
 * one granule probe together, which k_enc_probe caches in PROBE_CACHE = 24 rows before it sends the granule to the slow path.)
 * Clips whose step search runs past the step table (SURVEY A.E13) are outside the model: it stops with "overrun". */
#include "../../oracle/mp3stego_oracle.c"
#include <stdio.h>
static int g_slow, g_have; static int g_la[3]; static unsigned char g_seen[128]; static int g_nseen;
static int my_probe(enc_t*e,int32_t*ix,grinfo_t*ci,int step){ if(!g_seen[step+127]){g_seen[step+127]=1;g_nseen++;} int b=probe_bits(e,ix,ci); if(ci->big_values==0&&ci->count1>0&&!g_have) g_slow=1; if(ci->big_values>0){g_have=1;g_la[0]=ci->address1;g_la[1]=ci->address2;g_la[2]=ci->address3;} return b;}
static void run_variant(enc_t *e, grinfo_t ci0, int max_bits, const char *bits, int hn, grinfo_t *out, int *outbits)
{
    static int32_t ix[576];
    grinfo_t ci = ci0;
    const char *sv_s = e->hide_str; int64_t sv_l = e->hide_len, sv_o = e->hide_off;
    e->hide_str = bits; e->hide_len = hn; e->hide_off = 0;
    g_slow=0; g_have=0;
    int next=-120,count=120;
    do{int half=count/2,bit; int s=next+half;
       if(quantize(e,ix,s)>8192) bit=100000; else bit=my_probe(e,ix,&ci,s);
       if(bit<max_bits) count=half; else {next+=half;count-=half;}
    }while(count>1);
    ci.quantizerStepSize=next;
    int b;
    do{ while(ci.quantizerStepSize<0&&quantize(e,ix,ci.quantizerStepSize+1)>8192) ci.quantizerStepSize++;
        if(ci.quantizerStepSize>=0){printf("overrun\n");exit(0);}
        ci.quantizerStepSize++; b=my_probe(e,ix,&ci,ci.quantizerStepSize);
    }while(b>max_bits);
    e->hide_str=sv_s; e->hide_len=sv_l; e->hide_off=sv_o;
    *out=ci; *outbits=b;
}
int main(int argc,char**argv){
    int nfr=atoi(argv[2]); int br=atoi(argv[3]);
    FILE*f=fopen(argv[1],"rb"); int16_t*pcm=malloc((size_t)nfr*1152*2*2); if(fread(pcm,2,(size_t)nfr*1152*2,f)){} fclose(f);
    f=fopen(argv[4],"rb"); char*pay=malloc(1<<20); int64_t plen=fread(pay,1,1<<20,f); fclose(f);
    if(argc>5&&atoi(argv[5])>=0) plen=atoi(argv[5]);
    int sr=argc>6?atoi(argv[6]):44100;
    enc_t*e=calloc(1,sizeof*e);
    e->nch=2;e->samplerate=sr;e->bitrate=br;e->sr_index=sr==44100?0:sr==48000?1:2;
    e->buffer=pcm;e->buffer_len=(int64_t)nfr*1152*2;e->buffer_pos[0]=0;e->buffer_pos[1]=1;
    e->hide_str=pay;e->hide_len=plen;e->cache=0;e->cache_bits=32;
    for(int i=0;i<10000;i++) e->int2idx[i]=(int32_t)(sqrt(sqrt((double)i)*(double)i)-0.0946+0.5);
    double avg=(2.0*576/(double)sr)*(1000*(double)br/8.0);
    e->whole_slots_per_frame=(int)avg;e->frac_slots_per_frame=avg-(double)e->whole_slots_per_frame;e->slot_lag=-e->frac_slots_per_frame;
    e->side_info_len=288;
    /* emulated state */
    int st_a[2][2][3]={{{0}}}, st_step[2][2]={{0}}; int64_t off=0;
    long ngr=0,nslow=0,nsil=0,bad=0; int maxsteps=0;
    for(int fr=0;fr<nfr;fr++){
        if(e->frac_slots_per_frame!=0){e->padding=e->slot_lag<=(e->frac_slots_per_frame-1.0)?1:0;e->slot_lag+=e->padding-e->frac_slots_per_frame;}
        e->bits_per_frame=8*(e->whole_slots_per_frame+e->padding);
        e->mean_bits=(int)((e->bits_per_frame-e->side_info_len)/2.0);
        mdct_sub(e);
        for(int ch=0;ch<2;ch++)for(int gr=0;gr<2;gr++){
            int32_t*ix=e->l3_enc[ch][gr]; e->xr=e->mdct_freq[ch][gr]; e->xrmax=0;
            for(int i=575;i>=0;i--){e->xrsq[i]=e_mulsr(e->xr[i],e->xr[i]);int64_t ab=e->xr[i]<0?-(int64_t)e->xr[i]:(int64_t)e->xr[i];e->xrabs[i]=(int32_t)ab;if(e->xrabs[i]>e->xrmax)e->xrmax=e->xrabs[i];}
            grinfo_t*ci=&e->gi[gr][ch];
            int max_bits=e->mean_bits/2; if(max_bits>4095)max_bits=4095;
            ci->part2_3_length=0;ci->big_values=0;ci->count1=0;ci->table_select[0]=ci->table_select[1]=ci->table_select[2]=0;ci->region0_count=0;ci->region1_count=0;ci->count1table_select=0;
            ngr++;
            /* emulation */
            int em_ts[3]={0,0,0}, em_p23=0, em_bv=0,em_c1=0;
            if(e->xrmax){
                int q=2*ch+gr; int hiding=plen>0; int sure3=plen-3*(4*(int64_t)fr+q)>=3;
                grinfo_t rec[15]; int rbits[15]; int rhave[15]; int rla[15][3]; int slow=0;
                memset(g_seen,0,sizeof g_seen); g_nseen=0;
                for(int v=0;v<15;v++){
                    int active=hiding?(v<(sure3?8:15)):(v==14); if(!active) continue;
                    int hn; int hb; if(v<8){hn=3;hb=v;}else if(v<12){hn=2;hb=v-8;}else if(v<14){hn=1;hb=v-12;}else{hn=0;hb=0;}
                    char b[3]={(hb&1)?'1':'0',(hb&2)?'1':'0',(hb&4)?'1':'0'};
                    grinfo_t z=*ci; z.address1=z.address2=z.address3=0;
                    run_variant(e,z,max_bits,b,hn,&rec[v],&rbits[v]); if(g_slow) slow=1; rhave[v]=g_have; memcpy(rla[v],g_la,sizeof g_la);
                }
                if(g_nseen>maxsteps) maxsteps=g_nseen;
                /* resolve */
                int hn=0; int hb=0; if(hiding){int64_t left=plen-off; hn=left>3?3:(left<0?0:(int)left); for(int k=0;k<hn;k++) if(pay[off+k]=='1') hb|=1<<k;}
                int v=hn==3?hb:hn==2?8+hb:hn==1?12+hb:14;
                grinfo_t o; int ob;
                if(slow){ nslow++; grinfo_t z=*ci; z.address1=st_a[gr][ch][0];z.address2=st_a[gr][ch][1];z.address3=st_a[gr][ch][2];
                    char b[3]={(hb&1)?'1':'0',(hb&2)?'1':'0',(hb&4)?'1':'0'}; run_variant(e,z,max_bits,b,hn,&o,&ob);
                    st_a[gr][ch][0]=o.address1;st_a[gr][ch][1]=o.address2;st_a[gr][ch][2]=o.address3;
                } else { o=rec[v]; ob=rbits[v]; if(rhave[v]){st_a[gr][ch][0]=rla[v][0];st_a[gr][ch][1]=rla[v][1];st_a[gr][ch][2]=rla[v][2];} }
                st_step[gr][ch]=o.quantizerStepSize;
                em_ts[0]=o.table_select[0];em_ts[1]=o.table_select[1];em_ts[2]=o.table_select[2]; em_p23=ob; em_bv=o.big_values; em_c1=o.count1;
                off+=(em_ts[0]>0)+(em_ts[1]>0)+(em_ts[2]>0);
                /* real */
                ci->quantizerStepSize=bin_search_step_size(e,max_bits,ix,ci);
                int bits=inner_loop(e,ix,max_bits,ci);
                ci->part2_3_length=bits;
                e->hide_off+=(ci->table_select[0]>0)+(ci->table_select[1]>0)+(ci->table_select[2]>0);
            } else nsil++;
            int ok = em_ts[0]==ci->table_select[0]&&em_ts[1]==ci->table_select[1]&&em_ts[2]==ci->table_select[2]&&em_p23==ci->part2_3_length
                 &&em_bv==ci->big_values&&em_c1==ci->count1&&st_step[gr][ch]==ci->quantizerStepSize
                 &&st_a[gr][ch][0]==ci->address1&&st_a[gr][ch][1]==ci->address2&&st_a[gr][ch][2]==ci->address3&&off==e->hide_off;
            if(!ok){bad++; if(bad<5) printf("BAD fr %d ch %d gr %d: ts %d %d %d vs %d %d %d p23 %d vs %d a %d %d %d vs %d %d %d off %ld vs %ld\n",fr,ch,gr,em_ts[0],em_ts[1],em_ts[2],ci->table_select[0],ci->table_select[1],ci->table_select[2],em_p23,ci->part2_3_length,st_a[gr][ch][0],st_a[gr][ch][1],st_a[gr][ch][2],ci->address1,ci->address2,ci->address3,(long)off,(long)e->hide_off);}
        }
    }
    printf("granules %ld silent %ld slow %ld bad %ld maxsteps %d\n",ngr,nsil,nslow,bad,maxsteps);
    return 0;
}
